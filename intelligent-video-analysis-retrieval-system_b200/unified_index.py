"""``UnifiedIndex`` on the B200 path (boundary level B1).

Mirrors the search-side surface of the reference's ``unified_index.UnifiedIndex``
(unified_index.py:63-92, 480-538, 638-673, 1449-1459, 1755-1793, 1889-1938) with
the arithmetic moved to the sm_100a kernels behind ``faiss_compat.IndexFlatIP``.
An index is loaded either from an in-memory embedding matrix and metadata list
(``load_from_arrays`` / ``build_from_embeddings``) -- what the reference holds after
``_setup_memory_maps`` (``self.vectors``, ``self.metadata_list``, ``self.faiss_index``) --
or from a ``.rvdb`` file (``load_unified_index``, via ``rvdb_reader``: the vector, index
and metadata datasets only; thumbnails / images / checkpoints stay out of scope).

Result semantics reproduced on purpose (SURVEY.md section 0, fact 5):
``similarity_score = 1.0 - inner_product`` and ``rank`` is the 0-based position
in the FAISS result row (gaps allowed when hits are filtered).
"""
from __future__ import annotations

import threading
import time
from dataclasses import dataclass
from pathlib import Path
from typing import Any, Callable, Dict, List, Optional, Tuple

import numpy as np

from . import faiss_compat as faiss


@dataclass
class UnifiedIndexConfig:
    """Same fields and defaults as the reference dataclass (unified_index.py:49-60)."""
    compression_level: int = 6
    chunk_size: int = 1000
    memory_map: bool = True
    incremental_threshold: float = 0.1
    max_workers: int = 4
    image_quality: int = 95
    thumbnail_size: Tuple[int, int] = (224, 224)
    store_full_images: bool = False
    full_image_quality: int = 90


_BUILD_CHUNK = 10000      # rows normalised + added per step (unified_index.py:1770)


class UnifiedIndex:
    """Single-GPU unified index: exact top-k over L2-normalised keyframe embeddings."""

    def __init__(self, config: UnifiedIndexConfig = None, logger=None, device: int | None = None):
        self.config = config or UnifiedIndexConfig()
        self.logger = logger
        self.device = device
        self.is_loaded = False
        self.file_handle = None
        self.memory_maps: Dict[str, Dict] = {}
        self.vector_cache: Dict = {}
        self.metadata_cache: Dict[int, Dict] = {}
        self.faiss_index = None
        self.vectors = None
        self.metadata_list: List[Dict] = []
        self._folder_rows: Optional[Dict[str, np.ndarray]] = None
        self.lock = threading.RLock()

    # ------------------------------------------------------------------ build
    def build_from_embeddings(self, embeddings: np.ndarray, metadata_list: List[Dict],
                              normalize: bool = True, keep_vectors: bool = True) -> Dict[str, Any]:
        """The in-scope half of ``create_unified_index``: rows -> normalised -> index.

        Follows ``_build_faiss_index_from_file`` (unified_index.py:1755-1793):
        ``IndexFlatIP(dim)``; 10 000-row chunks, ``normalize_L2`` each, ``add``.
        """
        t0 = time.time()
        emb = np.asarray(embeddings)
        if emb.ndim != 2:
            raise ValueError("embeddings must be [n, d]")
        if len(metadata_list) != emb.shape[0]:
            raise ValueError(f"Features count ({emb.shape[0]}) != metadata count ({len(metadata_list)})")
        with self.lock:
            index = faiss.IndexFlatIP(emb.shape[1], device=self.device)
            index.reserve(emb.shape[0])
            for s in range(0, emb.shape[0], _BUILD_CHUNK):
                chunk = np.array(emb[s:s + _BUILD_CHUNK], dtype=np.float32, order="C", copy=True)
                if normalize:
                    faiss.normalize_L2(chunk)
                index.add(chunk)
            self.faiss_index = index
            self.vectors = emb if keep_vectors else None
            self.metadata_list = list(metadata_list)
            self.metadata_cache = {}
            self._folder_rows = None
            self.memory_maps = {"thumbnails": {}, "temporal": {}}
            self.is_loaded = True
        return {"processed_files": emb.shape[0], "vector_dim": emb.shape[1],
                "build_time": time.time() - t0}

    load_from_arrays = build_from_embeddings

    def create_unified_index(self, keyframes_dir: str, clip_processor, output_file: str = None,
                             csv_mappings: Dict[str, str] = None, progress_callback: Callable = None,
                             resume_from_existing: bool = False, chunk_size: int = 1000) -> Dict[str, Any]:
        """Index-build API (unified_index.py:94-363) restricted to the vector path.

        Scans ``keyframes_dir`` for ``*.jpg`` (sorted relative paths), embeds every
        image with ``clip_processor.encode_images([path], show_progress=False)[0]``
        (unified_index.py:828), builds the metadata dicts of unified_index.py:870-877
        and the GPU index.  Thumbnails, the .rvdb file, checkpoints and resume are
        out of scope; ``output_file`` is accepted and ignored.
        """
        import hashlib
        t0 = time.time()
        root = Path(keyframes_dir)
        files = sorted(root.rglob("*.jpg"), key=lambda p: str(p.relative_to(root)))
        vecs, metas, errors = [], [], []
        for n_done, p in enumerate(files):
            try:
                h = hashlib.sha256(p.read_bytes()).hexdigest()[:16]
                v = np.asarray(clip_processor.encode_images([str(p)], show_progress=False)[0], np.float32)
                try:
                    frame_id = int(p.stem)
                except ValueError:
                    frame_id = abs(hash(p.stem)) % 999999
                metas.append({"file_path": str(p), "folder_name": p.parts[-2] if len(p.parts) > 1 else "unknown",
                              "image_name": p.name, "frame_id": frame_id, "file_hash": h,
                              "file_size": p.stat().st_size})
                vecs.append(v)
            except Exception as e:           # reference: skip and record (unified_index.py:799-805)
                errors.append(f"{p}: {e}")
            if progress_callback:
                progress_callback(int((n_done + 1) / max(len(files), 1) * 80),
                                  f"Processing images... {n_done + 1}/{len(files)}")
        if not vecs:
            raise ValueError(f"no images could be processed under {keyframes_dir}")
        stats = self.build_from_embeddings(np.stack(vecs), metas)
        stats.update({"total_files": len(files), "skipped_files": len(files) - len(vecs),
                      "errors": errors, "build_time": time.time() - t0, "index_size": 0,
                      "compression_ratio": 1.0, "output_file": output_file})
        if progress_callback:
            progress_callback(100, "done")
        return stats

    def load_unified_index(self, index_file: str, load_vectors: bool = False) -> Dict[str, Any]:
        """Load a ``.rvdb`` file the way ``_setup_memory_maps`` does (unified_index.py:1175-1234), without h5py / lz4
        (``rvdb_reader``: HDF5 subset + LZ4 frame + LZF, bulk bytes decoded in C):

        * the index: the ``faiss_index`` dataset (raw bytes of ``faiss.write_index``) goes through
          ``faiss.deserialize_index`` exactly as in the reference (1182); older files keep it LZ4-framed under
          ``index/faiss`` (1185-1188); a file without either is indexed from its embeddings like
          ``_build_faiss_index_from_file`` (1755-1793: 10 000-row chunks, ``normalize_L2``, ``add``) -- the chunks are
          decoded and uploaded one after the other, the matrix is never assembled on the host;
        * the metadata list: ``metadata/data`` (LZ4 frame around JSON);
        * ``self.vectors``: the reference reads ALL embeddings into RAM here; searching does not need them, so they are
          read only on request (``load_vectors=True``)."""
        from . import rvdb_reader
        t0 = time.time()
        r = rvdb_reader.read_rvdb(index_file)
        try:
            emb = r["embeddings"]
            with self.lock:
                if r["faiss_index"] is not None:
                    index = faiss.deserialize_index(r["faiss_index"], device=self.device)
                elif emb is not None:
                    index = faiss.IndexFlatIP(emb.shape[1], device=self.device)
                    index.reserve(emb.shape[0])
                    expect = 0
                    for first, rows in emb.iter_row_blocks():
                        if first != expect:
                            raise rvdb_reader.RvdbFormatError(f"{index_file}: embedding chunks out of order")
                        for s in range(0, len(rows), _BUILD_CHUNK):
                            chunk = np.array(rows[s:s + _BUILD_CHUNK], dtype=np.float32, order="C", copy=True)
                            faiss.normalize_L2(chunk)
                            index.add(chunk)
                        expect += len(rows)
                else:
                    raise KeyError("FAISS index not found in file")
                self.faiss_index = index
                self.vectors = emb.read() if (load_vectors and emb is not None) else None
                self.metadata_list = r["metadata"]
                self.metadata_cache = {}
                self._folder_rows = None
                self.memory_maps = {"thumbnails": {}, "temporal": {}}
                self.is_loaded = True
        finally:
            r["file"].close()
        return {"load_time": time.time() - t0, "index_info": {"processed_files": len(self.metadata_list),
                                                               "vector_dim": self.faiss_index.d}}

    # ----------------------------------------------------------------- search
    def search_vectors(self, query_vector: np.ndarray, k: int = 50,
                       filter_func: Callable = None, videos=None) -> List[Dict[str, Any]]:
        """Drop-in for unified_index.py:480-538 (one query -> list of hit dicts).

        ``videos`` (folder names) takes the top-k on the GPU over the frames whose ``metadata["folder_name"]`` is one
        of them -- the k best frames of those videos, where ``filter_func`` can only drop hits from the global top-k.
        ``filter_func`` still applies afterwards; unknown names select nothing."""
        if not self.is_loaded:
            raise ValueError("Index not loaded. Call load_unified_index() first.")
        try:
            start = time.time()
            distances, indices = self._search(np.asarray(query_vector).reshape(1, -1), k, videos)
            results = []
            for i, (dist, idx) in enumerate(zip(distances[0], indices[0])):
                if idx == -1:
                    break
                metadata = self._get_metadata_cached(idx)
                if metadata is None:
                    continue
                if filter_func and not filter_func(metadata):
                    continue
                results.append({"rank": i, "similarity_score": float(1.0 - dist),
                                "metadata": metadata, "index": int(idx)})
            if self.logger:
                self.logger.debug(f"Search completed in {(time.time() - start) * 1000:.2f}ms, "
                                  f"found {len(results)} results")
            return results
        except Exception as e:
            if self.logger:
                self.logger.error(f"Search failed: {e}")
            raise

    def search_vectors_batch(self, query_vectors, k: int = 50,
                             filter_func: Callable = None, videos=None) -> List[List[Dict[str, Any]]]:
        """Many queries in ONE kernel call; element i equals ``search_vectors(query_vectors[i], k, filter_func,
        videos)``.

        The reference is strictly one query per call (unified_index.py:503; system.py:733-826 loops over
        queries); batching is where the tensor-core path pays off (SURVEY.md section 8f, rank 4)."""
        if not self.is_loaded:
            raise ValueError("Index not loaded. Call load_unified_index() first.")
        q = np.asarray(query_vectors)
        q = q.reshape(1, -1) if q.ndim == 1 else q.reshape(q.shape[0], -1)
        distances, indices = self._search(q, k, videos)
        out = []
        for drow, irow in zip(distances, indices):
            results = []
            for i, (dist, idx) in enumerate(zip(drow, irow)):
                if idx == -1:
                    break
                metadata = self._get_metadata_cached(idx)
                if metadata is None:
                    continue
                if filter_func and not filter_func(metadata):
                    continue
                results.append({"rank": i, "similarity_score": float(1.0 - dist),
                                "metadata": metadata, "index": int(idx)})
            out.append(results)
        return out

    def _search(self, q, k, videos):
        """``faiss_index.search(q, k)``, restricted to the rows of ``videos`` when given."""
        if videos is None:
            return self.faiss_index.search(q, k)
        sel = faiss.IDSelectorBatch(self.video_rows(videos))
        try:
            return self.faiss_index.search(q, k, params=faiss.SearchParameters(sel=sel))
        finally:
            sel.close()

    def video_rows(self, videos) -> np.ndarray:
        """Ascending row ids of the frames whose ``metadata["folder_name"]`` is in ``videos`` (a name or an iterable
        of names); unknown names contribute nothing.  The folder -> rows map is built once per loaded index."""
        if isinstance(videos, str):
            videos = [videos]
        with self.lock:
            if self._folder_rows is None:
                groups: Dict[str, List[int]] = {}
                for i, meta in enumerate(self.metadata_list):
                    name = meta.get("folder_name") if isinstance(meta, dict) else None
                    if name is not None:
                        groups.setdefault(name, []).append(i)
                self._folder_rows = {name: np.asarray(rows, np.int64) for name, rows in groups.items()}
            parts = [self._folder_rows[v] for v in set(videos) if v in self._folder_rows]
        return np.sort(np.concatenate(parts)) if parts else np.zeros(0, np.int64)

    # README facade (README.md:124-136): batched, raw inner products, metadata join
    def search(self, query, top_k: int = 10):
        """(ids int64[nq,k], scores float32[nq,k] descending inner product, metadata lists)."""
        if not self.is_loaded:
            raise ValueError("Index not loaded. Call load_unified_index() first.")
        q = np.asarray(query, dtype=np.float32)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        scores, ids = self.faiss_index.search(q, int(top_k))
        meta = [[self._get_metadata_cached(int(i)) if i >= 0 else None for i in row] for row in ids]
        return ids, scores, meta

    def augmented_search(self, query, top_k: int = 10, temporal_window: int = 3):
        """``search`` plus the temporal-context join (README.md:175-185)."""
        ids, scores, meta = self.search(query, top_k)
        ctx = [[self.get_temporal_context(int(i), temporal_window) if i >= 0 else [] for i in row]
               for row in ids]
        return ids, scores, meta, ctx

    # ------------------------------------------------------------------- join
    def _get_metadata_cached(self, index: int) -> Optional[Dict]:
        """unified_index.py:1449-1459."""
        index = int(index)
        if index in self.metadata_cache:
            return self.metadata_cache[index]
        if 0 <= index < len(self.metadata_list):
            metadata = self.metadata_list[index]
            self.metadata_cache[index] = metadata
            return metadata
        return None

    def get_temporal_context(self, frame_index: int, window_size: int = 5) -> List[int]:
        """unified_index.py:638-673 (pre-computed neighbours; empty unless populated)."""
        try:
            if not self.is_loaded:
                return []
            temporal = self.memory_maps.get("temporal", {})
            if frame_index in temporal:
                nb = temporal[frame_index]
                s = max(0, len(nb) // 2 - window_size)
                e = min(len(nb), len(nb) // 2 + window_size + 1)
                return nb[s:e]
            return []
        except Exception:
            return []

    def get_thumbnail(self, frame_index: int):
        return None            # image payloads are out of scope (SURVEY.md section 2)

    def get_full_image(self, frame_index: int):
        return None

    def get_statistics(self) -> Dict[str, Any]:
        return {"is_loaded": self.is_loaded,
                "ntotal": self.faiss_index.ntotal if self.faiss_index is not None else 0,
                "metadata_entries": len(self.metadata_list),
                "metadata_cache_size": len(self.metadata_cache)}

    # -------------------------------------------------------------- lifecycle
    def close(self):
        with self.lock:
            if self.faiss_index is not None and hasattr(self.faiss_index, "close"):
                self.faiss_index.close()
            self.faiss_index = None
            self.is_loaded = False
            self.metadata_cache.clear()
            self.vector_cache.clear()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False


def create_optimized_index(keyframes_dir: str, clip_processor, output_file: str,
                           csv_mappings: Dict[str, str] = None, config: UnifiedIndexConfig = None,
                           logger=None, progress_callback: Callable = None,
                           resume_from_existing: bool = False, chunk_size: int = 1000) -> Dict[str, Any]:
    """unified_index.py:1889-1919 (the index stays open: it lives in HBM, not in a file)."""
    unified_index = UnifiedIndex(config, logger)
    stats = unified_index.create_unified_index(keyframes_dir, clip_processor, output_file, csv_mappings,
                                               progress_callback, resume_from_existing, chunk_size)
    stats["index"] = unified_index
    return stats


def load_optimized_index(index_file: str, config: UnifiedIndexConfig = None, logger=None) -> UnifiedIndex:
    """unified_index.py:1922-1938."""
    unified_index = UnifiedIndex(config, logger)
    unified_index.load_unified_index(index_file)
    return unified_index
