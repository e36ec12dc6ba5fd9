"""ctypes binding of liboramacore_b200.so (the C ABI in include/oramacore_b200.h).

The library is CUDA-only.  Loading succeeds on a CPU box (symbols resolve; used by the
`not gpu` tests), every compute call fails loudly with OcError when no sm_100 device is
present — there is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("OC_SO_PATH") or os.path.join(_HERE, "liboramacore_b200.so")   # OC_SO_PATH: A/B builds (csrc/Makefile)
CSRC = os.path.join(_HERE, "csrc")

OC_OK = 0
OC_MAX_TOPK = 1024
OC_COMM_ID_BYTES = 128

EXPORTED_SYMBOLS = [
    "oc_last_error", "oc_version", "oc_abi_sizes", "oc_init", "oc_shutdown", "oc_device_info", "oc_comm_unique_id",
    "oc_comm_init", "oc_comm_p2p_export", "oc_comm_p2p_import", "oc_emb_create", "oc_emb_destroy", "oc_emb_reserve", "oc_emb_insert", "oc_emb_delete",
    "oc_emb_info", "oc_emb_search", "oc_str_create", "oc_str_destroy", "oc_str_set_rows", "oc_str_load_field",
    "oc_str_insert", "oc_str_commit", "oc_str_delete", "oc_str_info", "oc_str_set_global", "oc_search", "oc_pinned_alloc", "oc_pinned_free", "oc_last_timing", "oc_launch_count",
    "oc_batcher_create", "oc_batcher_destroy", "oc_batcher_search", "oc_batcher_stats",
    "oc_filter_from_ids", "oc_filter_from_bits", "oc_filter_and", "oc_filter_or", "oc_filter_not", "oc_filter_count",
    "oc_filter_read", "oc_filter_destroy", "oc_merge_results",
    "oc_facets_create", "oc_facets_destroy", "oc_facets_add_field", "oc_facets_add_number_field", "oc_search_facets",
    "oc_sort_create", "oc_sort_destroy", "oc_sort_add_number_field", "oc_sort_add_date_field", "oc_sort_add_bool_field",
    "oc_search_sorted", "oc_sort_last_forms", "oc_merge_sorted_results",
    "oc_dict_create", "oc_dict_destroy", "oc_dict_add_terms", "oc_dict_lookup", "oc_dict_size", "oc_dict_set_stemmer", "oc_stem_english",
    "oc_dict_resolve", "oc_resolved_arrays", "oc_resolved_fill", "oc_resolved_free",
]


class OcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"oramacore_b200 error {code}: {msg}")
        self.code = code


class EmbInfo(C.Structure):
    _fields_ = [("num_embeddings", C.c_uint64), ("num_rows", C.c_uint64), ("dimensions", C.c_uint32),
                ("dtype", C.c_int), ("device_bytes", C.c_uint64)]


class StrInfo(C.Structure):
    _fields_ = [("total_documents", C.c_uint64), ("total_postings", C.c_uint64),
                ("unique_terms_count", C.c_uint64), ("n_fields", C.c_uint32), ("device_bytes", C.c_uint64),
                ("version", C.c_uint64), ("pending_postings", C.c_uint64)]


class SearchParams(C.Structure):
    _fields_ = [("mode", C.c_int), ("n_queries", C.c_uint32), ("limit", C.c_uint32), ("offset", C.c_uint32),
                ("similarity", C.c_float), ("threshold", C.c_float), ("bm25_k", C.c_float), ("bm25_b", C.c_float),
                ("q_vecs", C.c_void_p), ("q_token_offsets", C.c_void_p), ("token_term_offsets", C.c_void_p),
                ("term_field", C.c_void_p), ("term_id", C.c_void_p), ("term_weight", C.c_void_p),
                ("filter_bits", C.c_void_p), ("filter_nbits", C.c_uint64),
                ("omc_doc_ids", C.c_void_p), ("omc_mult", C.c_void_p), ("n_omc", C.c_uint64),
                ("sharded", C.c_int), ("vector_limit", C.c_uint32), ("filter", C.c_void_p)]


class FacetReq(C.Structure):
    _fields_ = [("field", C.c_uint32), ("variant", C.c_uint32), ("from_", C.c_double), ("to", C.c_double)]


class ResolveParams(C.Structure):
    _fields_ = [("texts", C.POINTER(C.c_char_p)), ("n_queries", C.c_uint32), ("exact", C.c_int), ("tolerance", C.c_int),
                ("field_boost", C.c_void_p), ("field_mask", C.c_void_p), ("exact_match_boost", C.c_float)]


STEM_FN = C.CFUNCTYPE(C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p)


class Timing(C.Structure):
    _fields_ = [("h2d_ms", C.c_float), ("device_ms", C.c_float), ("d2h_ms", C.c_float), ("scan_ms", C.c_float),
                ("bm25_ms", C.c_float), ("fuse_ms", C.c_float), ("comm_ms", C.c_float),
                ("kernel_launches", C.c_uint32), ("scan_launches", C.c_uint32), ("scan_bytes", C.c_uint64),
                ("bm25_postings", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("scan_tensor_core", C.c_uint32), ("scan_unproven", C.c_uint32),
                ("scan_variant", C.c_uint32), ("scan_sweep_ms", C.c_float), ("rerun_ms", C.c_float),
                ("scan_rescored", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


def build(force: bool = False) -> str:
    """Compile the shared library in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    srcs.append(os.path.join(_HERE, "..", "include", "oramacore_b200.h"))
    stale = (not os.path.exists(SO_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(SO_PATH) for s in srcs)
    if force or stale:
        r = subprocess.run(["make", "-C", CSRC] + (["-B"] if force else []), capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc build failed:\n" + r.stdout + r.stderr)
    return SO_PATH


_lib = None


def lib():
    """Load the CUDA library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise OcError(-2, f"{SO_PATH} is missing: run __graft_entry__.build() (nvcc, sm_100a). "
                          "There is no CPU fallback.")
    L = C.CDLL(SO_PATH)
    vp, u32, u64, f32, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_float, C.c_int
    L.oc_last_error.restype = C.c_char_p
    L.oc_version.restype = i32
    L.oc_abi_sizes.argtypes = [C.POINTER(C.c_size_t)]
    L.oc_abi_sizes.restype = None
    L.oc_init.argtypes = [i32, C.POINTER(vp)]
    L.oc_shutdown.argtypes = [vp]
    L.oc_shutdown.restype = None
    L.oc_device_info.argtypes = [vp, C.POINTER(i32), C.POINTER(C.c_size_t), C.c_char_p, C.c_size_t]
    L.oc_comm_unique_id.argtypes = [vp]
    L.oc_comm_init.argtypes = [vp, i32, i32, vp]
    L.oc_comm_p2p_export.argtypes = [vp, vp]
    L.oc_comm_p2p_import.argtypes = [vp, vp]
    L.oc_emb_create.argtypes = [vp, u32, i32, i32, C.POINTER(vp)]
    L.oc_emb_destroy.argtypes = [vp]
    L.oc_emb_destroy.restype = None
    L.oc_emb_reserve.argtypes = [vp, u64]
    L.oc_emb_insert.argtypes = [vp, vp, vp, u64]
    L.oc_emb_delete.argtypes = [vp, vp, u64]
    L.oc_emb_info.argtypes = [vp, C.POINTER(EmbInfo)]
    L.oc_emb_search.argtypes = [vp, vp, u32, u32, f32, vp, u64, vp, vp, vp]
    L.oc_str_create.argtypes = [vp, u32, C.POINTER(vp)]
    L.oc_str_destroy.argtypes = [vp]
    L.oc_str_destroy.restype = None
    L.oc_str_set_rows.argtypes = [vp, u64, vp, u64]
    L.oc_str_load_field.argtypes = [vp, u32, f32, u32, vp, vp, vp, vp, vp]
    L.oc_str_insert.argtypes = [vp, u32, u64, C.c_uint16, u32, vp, vp]
    L.oc_str_commit.argtypes = [vp]
    L.oc_str_set_global.argtypes = [vp, u64, vp]
    L.oc_str_delete.argtypes = [vp, vp, u64]
    L.oc_str_info.argtypes = [vp, C.POINTER(StrInfo)]
    L.oc_search.argtypes = [vp, vp, vp, C.POINTER(SearchParams), vp, vp, vp, vp]
    L.oc_batcher_create.argtypes = [vp, vp, vp, u32, u32, C.POINTER(vp)]
    L.oc_batcher_destroy.argtypes = [vp]
    L.oc_batcher_destroy.restype = None
    L.oc_batcher_search.argtypes = [vp, C.POINTER(SearchParams), vp, vp, vp, vp]
    L.oc_batcher_stats.argtypes = [vp, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64)]
    L.oc_filter_from_ids.argtypes = [vp, vp, u64, u64, C.POINTER(vp)]
    L.oc_filter_from_bits.argtypes = [vp, vp, u64, C.POINTER(vp)]
    L.oc_filter_and.argtypes = [vp, vp, C.POINTER(vp)]
    L.oc_filter_or.argtypes = [vp, vp, C.POINTER(vp)]
    L.oc_filter_not.argtypes = [vp, C.POINTER(vp)]
    L.oc_filter_count.argtypes = [vp, C.POINTER(u64)]
    L.oc_filter_read.argtypes = [vp, vp]
    L.oc_filter_destroy.argtypes = [vp]
    L.oc_filter_destroy.restype = None
    L.oc_facets_create.argtypes = [vp, u64, C.POINTER(vp)]
    L.oc_facets_destroy.argtypes = [vp]
    L.oc_facets_destroy.restype = None
    L.oc_facets_add_field.argtypes = [vp, u32, vp, vp, C.POINTER(u32)]
    L.oc_facets_add_number_field.argtypes = [vp, u64, vp, vp, C.POINTER(u32)]
    L.oc_search_facets.argtypes = [vp, vp, vp, vp, C.POINTER(SearchParams), C.POINTER(FacetReq), u32, vp]
    L.oc_merge_results.argtypes = [u32, u32, u32, u32, u32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), vp, vp, vp, vp]
    L.oc_sort_create.argtypes = [vp, u64, C.POINTER(vp)]
    L.oc_sort_destroy.argtypes = [vp]
    L.oc_sort_destroy.restype = None
    L.oc_sort_add_number_field.argtypes = [vp, u64, vp, vp, C.POINTER(u32)]
    L.oc_sort_add_date_field.argtypes = [vp, u64, vp, vp, C.POINTER(u32)]
    L.oc_sort_add_bool_field.argtypes = [vp, u64, vp, u64, vp, C.POINTER(u32)]
    L.oc_search_sorted.argtypes = [vp, vp, vp, vp, u32, i32, C.POINTER(SearchParams), vp, vp, vp, vp, vp]
    L.oc_sort_last_forms.argtypes = [vp, u32, vp]
    L.oc_merge_sorted_results.argtypes = [u32, u32, u32, u32, u32, i32] + [C.POINTER(vp)] * 5 + [vp, vp, vp, vp]
    L.oc_dict_create.argtypes = [u32, C.POINTER(vp)]
    L.oc_dict_destroy.argtypes = [vp]
    L.oc_dict_destroy.restype = None
    L.oc_dict_add_terms.argtypes = [vp, u32, C.POINTER(C.c_char_p), u32, vp]
    L.oc_dict_lookup.argtypes = [vp, u32, C.c_char_p, C.POINTER(u32)]
    L.oc_dict_size.argtypes = [vp, u32]
    L.oc_dict_size.restype = u32
    L.oc_dict_set_stemmer.argtypes = [vp, vp, vp]
    L.oc_stem_english.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, vp]
    L.oc_stem_english.restype = C.c_size_t
    L.oc_dict_resolve.argtypes = [vp, C.POINTER(ResolveParams), C.POINTER(vp)]
    L.oc_resolved_arrays.argtypes = [vp] + [C.POINTER(vp)] * 5 + [C.POINTER(u32)] * 2
    L.oc_resolved_arrays.restype = None
    L.oc_resolved_fill.argtypes = [vp, C.POINTER(SearchParams)]
    L.oc_resolved_fill.restype = None
    L.oc_resolved_free.argtypes = [vp]
    L.oc_resolved_free.restype = None
    L.oc_pinned_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.oc_pinned_free.argtypes = [vp]
    L.oc_pinned_free.restype = None
    L.oc_last_timing.argtypes = [vp, C.POINTER(Timing)]
    L.oc_launch_count.argtypes = [vp]
    L.oc_launch_count.restype = u64
    _lib = L
    return L


def check(rc: int):
    if rc != OC_OK:
        raise OcError(rc, lib().oc_last_error().decode("utf-8", "replace"))
