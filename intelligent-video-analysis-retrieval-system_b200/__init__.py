"""B200-native retrieval hot path of Intelligent-Video-Analysis-Retrieval-System.

Exact top-k inner-product search over L2-normalised keyframe embeddings and
windowed near-duplicate keyframe pruning, as hand-written sm_100a CUDA kernels
behind a C ABI (include/ivr_b200.h), with the reference's Python call
signatures on top.  Importing this package loads ``libivr_b200.so``; there is
no CPU fallback.

The directory name contains hyphens; import it through the ``ivr_b200`` alias
module at the repository root (``import ivr_b200``).
"""
from . import _native, faiss_compat, frame_filter, sharded           # noqa: F401
from .facade import RAGBuilder, RAGRetriever                          # noqa: F401
from .faiss_compat import (IDSelectorBatch, IDSelectorBitmap, IDSelectorNot, IDSelectorRange,  # noqa: F401
                           IndexFlatIP, SearchParameters, normalize_L2)
from .frame_filter import FrameFilter                                 # noqa: F401
from .relationships import build_similarity_relationships            # noqa: F401
from .retriever import FAISSRetriever, KeyframeMetadata, SearchResult  # noqa: F401
from .sharded import ShardedFlatIP                                    # noqa: F401
from .temporal import TemporalAnalyzer                                # noqa: F401
from .unified_builder import UnifiedBuilderIntegration, add_unified_index_support  # noqa: F401
from .unified_index import (UnifiedIndex, UnifiedIndexConfig, create_optimized_index,  # noqa: F401
                            load_optimized_index)

__version__ = "0.1.0"
