"""oramacore_b200 — B200-native (sm_100a) implementation of OramaCore's search hot path:
embedding scan + BM25F posting scorer + hybrid fusion/top-k behind the reference's
search() surface (mode = fulltext | vector | hybrid).  CUDA only; no CPU fallback."""
from .types import (FieldPostings, StringIndexData, TextQuery, SearchHits, MODE_FULLTEXT, MODE_VECTOR,
                    MODE_HYBRID, BM25_B, BM25_K)
from ._lib import OcError, build, lib, SO_PATH
from .engine import (Context, DeviceFilter, FacetStore, SortStore, merge_index_results, merge_sorted_index_results, search_facets, search_sorted, EmbeddingFieldStorage, SearchBatcher, StringFieldStorage, TermDictionary, TextQueryBatch, TokenScoreContext, TokenScoreParams,
                     VectorSearchParams, from_bf16, pinned_empty, search, to_bf16)

__all__ = ["FieldPostings", "StringIndexData", "TextQuery", "SearchHits", "MODE_FULLTEXT", "MODE_VECTOR",
           "MODE_HYBRID", "BM25_B", "BM25_K", "OcError", "build", "lib", "SO_PATH", "Context", "DeviceFilter", "FacetStore", "SortStore", "merge_index_results", "merge_sorted_index_results", "search_facets", "search_sorted",
           "EmbeddingFieldStorage", "SearchBatcher", "StringFieldStorage", "TermDictionary", "TextQueryBatch", "TokenScoreContext", "TokenScoreParams",
           "VectorSearchParams", "from_bf16", "pinned_empty", "search", "to_bf16"]
