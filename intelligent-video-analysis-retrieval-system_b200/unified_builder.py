"""``UnifiedBuilderIntegration`` on the B200 path (boundary level B1).

Mirrors unified_builder.py:26-440.  ``system.unified_builder`` is a duck-typed
slot in the reference (system.py:1691, 804-807; gui.py:5520): anything with a
truthy ``.unified_index`` (having ``.is_loaded``) and
``.search_unified_fast(q, k, thr)`` is used, so an instance of this class can be
installed there directly (INTEGRATION.md).
"""
from __future__ import annotations

import time
from typing import Any, Callable, Dict, List, Optional

import numpy as np

from .retriever import KeyframeMetadata
from .unified_index import UnifiedIndex, UnifiedIndexConfig


class UnifiedBuilderIntegration:
    def __init__(self, system=None, logger=None, device: int | None = None):
        self.system = system
        self.logger = logger if logger is not None else getattr(system, "logger", None)
        self.unified_index: Optional[UnifiedIndex] = None
        self.device = device

    # ---- build / load -----------------------------------------------------
    def create_unified_index_fast(self, keyframes_dir: str, output_path: str = None,
                                  csv_mappings: Dict[str, str] = None,
                                  progress_callback: Callable = None,
                                  resume_from_existing: bool = False,
                                  chunk_size: int = 1000) -> Dict[str, Any]:
        """unified_builder.py:39-133 (vector path; the index is left loaded in HBM)."""
        start = time.time()
        if output_path is None:
            output_path = f"unified_index_{int(time.time())}.rvdb"
        if not getattr(self.system, "clip_processor", None) and hasattr(self.system, "_initialize_ai_components"):
            self.system._initialize_ai_components()
        config = UnifiedIndexConfig(compression_level=6, chunk_size=2000, memory_map=True, max_workers=4,
                                    image_quality=95, thumbnail_size=(224, 224), store_full_images=True,
                                    full_image_quality=90)
        self.unified_index = UnifiedIndex(config, self.logger, device=self.device)
        stats = self.unified_index.create_unified_index(
            keyframes_dir, self.system.clip_processor, output_path, csv_mappings, progress_callback,
            resume_from_existing, chunk_size)
        stats["total_build_time"] = time.time() - start
        stats["output_file"] = output_path
        old = stats["processed_files"] * 0.05
        speedup = old / stats["build_time"] if stats["build_time"] > 0 else 1.0
        stats["estimated_speedup"] = f"{speedup:.1f}x faster than legacy system"
        return stats

    def load_unified_index_fast(self, index_file: str) -> Dict[str, Any]:
        """unified_builder.py:135-188."""
        start = time.time()
        self.unified_index = UnifiedIndex(UnifiedIndexConfig(memory_map=True), self.logger, device=self.device)
        load_stats = self.unified_index.load_unified_index(index_file)
        load_stats["total_load_time"] = time.time() - start
        return load_stats

    def load_from_arrays(self, embeddings: np.ndarray, metadata_list: List[Dict]) -> Dict[str, Any]:
        """In-memory equivalent of ``load_unified_index_fast`` (no .rvdb container)."""
        self.unified_index = UnifiedIndex(UnifiedIndexConfig(memory_map=True), self.logger, device=self.device)
        return self.unified_index.build_from_embeddings(embeddings, metadata_list)

    # ---- search (unified_builder.py:190-251) ------------------------------
    def search_unified_fast(self, query_vector: "np.ndarray", k: int = 50,
                            similarity_threshold: float = 0.0, videos=None) -> List[Dict[str, Any]]:
        """``videos``: restrict the top-k to those folder names (``UnifiedIndex.search_vectors``)."""
        if not self.unified_index:
            raise ValueError("Unified index not loaded. Call load_unified_index_fast() first.")
        results = self.unified_index.search_vectors(query_vector, k=k, filter_func=lambda meta: True, videos=videos)
        enriched = []
        for result in results:
            if result["similarity_score"] >= similarity_threshold:
                temporal = self.unified_index.get_temporal_context(result["index"], window_size=3)
                enriched.append({
                    "metadata": self._convert_metadata_to_legacy(result["metadata"]),
                    "similarity_score": result["similarity_score"],
                    "rank": result["rank"],
                    "temporal_context": temporal,
                    "index": result["index"],
                })
        return enriched

    def search_unified_fast_batch(self, query_vectors, k: int = 50,
                                  similarity_threshold: float = 0.0, videos=None) -> List[List[Dict[str, Any]]]:
        """``search_unified_fast`` for a batch of queries in one kernel call (same per-query result)."""
        if not self.unified_index:
            raise ValueError("Unified index not loaded. Call load_unified_index_fast() first.")
        batches = self.unified_index.search_vectors_batch(query_vectors, k=k, filter_func=lambda meta: True,
                                                          videos=videos)
        out = []
        for results in batches:
            enriched = []
            for result in results:
                if result["similarity_score"] >= similarity_threshold:
                    enriched.append({
                        "metadata": self._convert_metadata_to_legacy(result["metadata"]),
                        "similarity_score": result["similarity_score"],
                        "rank": result["rank"],
                        "temporal_context": self.unified_index.get_temporal_context(result["index"], window_size=3),
                        "index": result["index"],
                    })
            out.append(enriched)
        return out

    def get_thumbnail_fast(self, frame_index: int):
        return self.unified_index.get_thumbnail(frame_index) if self.unified_index else None

    def get_full_image_fast(self, frame_index: int):
        return self.unified_index.get_full_image(frame_index) if self.unified_index else None

    def incremental_update_fast(self, keyframes_dir: str, progress_callback: Callable = None):
        raise NotImplementedError("incremental .rvdb updates are file I/O (out of scope); "
                                  "append rows with unified_index.faiss_index.add instead")

    def get_index_stats(self) -> Dict[str, Any]:
        if not self.unified_index:
            return {"loaded": False}
        s = self.unified_index.get_statistics()
        s["loaded"] = True
        return s

    def close(self):
        if self.unified_index:
            self.unified_index.close()
            self.unified_index = None

    @staticmethod
    def _convert_metadata_to_legacy(metadata: Dict):
        """unified_builder.py:390-404: dict -> KeyframeMetadata, dict on failure."""
        try:
            return KeyframeMetadata(folder_name=metadata.get("folder_name", ""),
                                    image_name=metadata.get("image_name", ""),
                                    frame_id=metadata.get("frame_id", 0),
                                    file_path=metadata.get("file_path", ""))
        except Exception:
            return metadata


def add_unified_index_support(system_instance):
    """unified_builder.py:427-440."""
    if not hasattr(system_instance, "unified_builder"):
        system_instance.unified_builder = UnifiedBuilderIntegration(system_instance)
    return system_instance.unified_builder
