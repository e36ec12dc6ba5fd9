"""Host-side mirror of the reference's read-side scoring interface over the C ABI.

Names and argument meaning follow the reference (oramasearch/oramacore @ 666ab48):
  * EmbeddingFieldStorage  — read/index/embedding_field.rs:29-34 (insert :232, delete :240,
                             search :250-278, info/stats :303-310)
  * VectorSearchParams     — read/index/committed_field/vector.rs:10-15
  * StringFieldStorage set — read/index/string_field.rs (one oc_str per Index)
  * TokenScoreParams / TokenScoreContext.execute — read/index/token_score.rs:31-41, 460-509
  * search()               — the CollectionManager search surface restricted to the hot path
                             (read/search.rs:283-501): mode = fulltext | vector | hybrid.
All compute happens in liboramacore_b200.so on the GPU; nothing here scores on the CPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import OcError, SearchParams, Timing, check, lib
from .types import (BM25_B, BM25_K, MODE_FULLTEXT, MODE_HYBRID, MODE_VECTOR, SearchHits, StringIndexData,
                    TextQuery)

# Model::dimensions / rescale_score (python/embeddings.rs:52-92)
MODEL_DIMS = {
    "BGESmall": 384, "BGEBase": 768, "BGELarge": 1024, "JinaEmbeddingsV2BaseCode": 768,
    "MultilingualE5Small": 384, "MultilingualE5Base": 768, "MultilingualE5Large": 1024,
    "MultilingualMiniLML12V2": 384,
}
E5_MODELS = {"MultilingualE5Small", "MultilingualE5Base", "MultilingualE5Large"}


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    """One GPU + stream + workspace (oc_ctx). One per process, like one rank per GPU."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        check(lib().oc_init(device, C.byref(self._h)))
        self.device = device

    def close(self):
        if self._h:
            lib().oc_shutdown(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def device_info(self):
        sm = C.c_int()
        mem = C.c_size_t()
        name = C.create_string_buffer(256)
        check(lib().oc_device_info(self._h, C.byref(sm), C.byref(mem), name, 256))
        return {"sm_count": sm.value, "hbm_bytes": mem.value, "name": name.value.decode()}

    def last_timing(self) -> dict:
        t = Timing()
        check(lib().oc_last_timing(self._h, C.byref(t)))
        return t.as_dict()

    def launch_count(self) -> int:
        return int(lib().oc_launch_count(self._h))

    # ---- document-sharded multi-GPU (SURVEY.md §8e)
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (C.c_uint8 * _lib.OC_COMM_ID_BYTES)()
        check(lib().oc_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, world_size: int, rank: int, unique_id: bytes):
        buf = (C.c_uint8 * _lib.OC_COMM_ID_BYTES).from_buffer_copy(unique_id)
        check(lib().oc_comm_init(self._h, world_size, rank, buf))

    def comm_enable_p2p(self, all_gather):
        """Direct NVLink exchange of the shard records (oc_comm_p2p_*).  `all_gather(blob: bytes) -> list[bytes]`
        is the host runtime's all-gather in rank order (e.g. torch.distributed.all_gather_object)."""
        buf = (C.c_uint8 * 128)()
        check(lib().oc_comm_p2p_export(self._h, buf))
        blobs = all_gather(bytes(buf))
        cat = b"".join(blobs)
        arr = (C.c_uint8 * len(cat)).from_buffer_copy(cat)
        check(lib().oc_comm_p2p_import(self._h, arr))


def to_bf16(x: np.ndarray) -> np.ndarray:
    """fp32 -> bf16 bit patterns (uint16), round to nearest even."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32)
    r = u + np.uint32(0x7fff) + ((u >> np.uint32(16)) & np.uint32(1))
    return (r >> np.uint32(16)).astype(np.uint16)


def from_bf16(b: np.ndarray) -> np.ndarray:
    """bf16 bit patterns -> the fp32 values they denote (exact)."""
    return (b.astype(np.uint32) << np.uint32(16)).view(np.float32)


def pinned_empty(shape, dtype=np.float32) -> np.ndarray:
    """numpy array backed by page-locked host memory (oc_pinned_alloc): inputs placed here are DMA'd
    directly by oc_search. The memory is intentionally never freed before interpreter exit."""
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    check(lib().oc_pinned_alloc(n, C.byref(p)))
    buf = (C.c_uint8 * max(n, 1)).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


@dataclass
class VectorSearchParams:
    """committed_field/vector.rs:10-15"""
    target: np.ndarray
    similarity: float
    limit: int
    filtered_doc_ids: Optional[np.ndarray] = None  # bitmap over DocumentId (uint64 words)
    filter_nbits: int = 0


class EmbeddingFieldStorage:
    """embedding_field.rs:29-34 — cosine metric, device resident."""

    def __init__(self, ctx: Context, model: str = "BGEBase", dim: Optional[int] = None, dtype: str = "f32"):
        """dtype "f32" (what the reference stores, embedding_field.rs:232) or "bf16" (storage extension:
        rows are kept as bf16, scores are exact fp32 arithmetic on those values)."""
        self.ctx = ctx
        self.model = model
        self.dim = int(dim if dim is not None else MODEL_DIMS[model])
        self.dtype = dtype
        self._h = C.c_void_p()
        check(lib().oc_emb_create(ctx._h, self.dim, {"f32": 0, "bf16": 1}[dtype], 1 if model in E5_MODELS else 0,
                                  C.byref(self._h)))

    def close(self):
        if self._h:
            lib().oc_emb_destroy(self._h)
            self._h = C.c_void_p()

    def reserve(self, n_rows: int):
        check(lib().oc_emb_reserve(self._h, n_rows))

    def insert(self, doc_id: int, vectors: Sequence[Sequence[float]]):
        """insert(DocumentId, Vec<Vec<f32>>) — several chunks per document (embedding_field.rs:232-237)."""
        v = np.ascontiguousarray(np.asarray(vectors, np.float32).reshape(-1, self.dim))
        self.insert_batch(np.full(v.shape[0], doc_id, np.uint64), v)

    def insert_batch(self, doc_ids: np.ndarray, rows: np.ndarray):
        d = np.ascontiguousarray(doc_ids, np.uint64)
        if self.dtype == "bf16":   # fp32 input is rounded to bf16 (RNE); uint16 input is taken as bf16 bits
            r = np.ascontiguousarray(rows) if rows.dtype == np.uint16 else to_bf16(rows)
        else:
            r = np.ascontiguousarray(rows, np.float32)
        assert r.ndim == 2 and r.shape[1] == self.dim and r.shape[0] == d.shape[0]
        check(lib().oc_emb_insert(self._h, _p(d), _p(r), d.shape[0]))

    def delete(self, doc_id):
        """One DocumentId or a sequence of them."""
        d = np.ascontiguousarray(np.atleast_1d(np.asarray(doc_id, np.uint64)).ravel())
        check(lib().oc_emb_delete(self._h, _p(d), int(d.shape[0])))

    def info(self) -> dict:
        i = _lib.EmbInfo()
        check(lib().oc_emb_info(self._h, C.byref(i)))
        return {"num_embeddings": i.num_embeddings, "num_rows": i.num_rows, "dimensions": i.dimensions,
                "device_bytes": i.device_bytes}

    def search_batch(self, targets: np.ndarray, limit: int, similarity: float,
                     filter_bits: Optional[np.ndarray] = None, filter_nbits: int = 0):
        q = np.ascontiguousarray(targets, np.float32).reshape(-1, self.dim)
        B = q.shape[0]
        docs = np.zeros((B, limit), np.uint64)
        scores = np.zeros((B, limit), np.float32)
        counts = np.zeros(B, np.uint32)
        fb = None if filter_bits is None else np.ascontiguousarray(filter_bits, np.uint64)
        check(lib().oc_emb_search(self._h, _p(q), B, limit, similarity, _p(fb), int(filter_nbits),
                                  _p(docs), _p(scores), _p(counts)))
        return docs, scores, counts

    def search(self, params: VectorSearchParams, output: Dict[int, float]) -> None:
        """EmbeddingFieldStorage::search(&VectorSearchParams, &mut HashMap) — `output[doc] += score`."""
        docs, scores, counts = self.search_batch(params.target, params.limit, params.similarity,
                                                 params.filtered_doc_ids, params.filter_nbits)
        for i in range(int(counts[0])):
            d = int(docs[0, i])
            output[d] = np.float32(output.get(d, np.float32(0.0)) + scores[0, i])


class StringFieldStorage:
    """All string fields of one Index on the device (string_field.rs:32-36); built from
    committed postings (`StringIndexData`)."""

    def __init__(self, ctx: Context, data: StringIndexData, global_df: Optional[List[np.ndarray]] = None):
        self.ctx = ctx
        self.data = data
        self._h = C.c_void_p()
        check(lib().oc_str_create(ctx._h, len(data.fields), C.byref(self._h)))
        rd = None if data.row_doc_ids is None else np.ascontiguousarray(data.row_doc_ids, np.uint64)
        check(lib().oc_str_set_rows(self._h, int(data.n_rows), _p(rd), int(data.document_count)))
        for i, f in enumerate(data.fields):
            f.validate()
            gdf = None if global_df is None else np.ascontiguousarray(global_df[i], np.uint32)
            check(lib().oc_str_load_field(self._h, i, float(f.avg_field_len), f.n_terms,
                                          _p(np.ascontiguousarray(f.term_offsets)), _p(np.ascontiguousarray(f.post_row)),
                                          _p(np.ascontiguousarray(f.post_tf)), _p(np.ascontiguousarray(f.post_len)),
                                          _p(gdf)))

    @classmethod
    def empty(cls, ctx: Context, n_fields: int = 1) -> "StringFieldStorage":
        """StringFieldStorage::new (string_field.rs:72-82): no committed postings yet."""
        self = cls.__new__(cls)
        self.ctx, self.data = ctx, None
        self._h = C.c_void_p()
        check(lib().oc_str_create(ctx._h, n_fields, C.byref(self._h)))
        return self

    def close(self):
        if self._h:
            lib().oc_str_destroy(self._h)
            self._h = C.c_void_p()

    def insert(self, doc_id: int, field: int, field_length: int, terms: Dict[int, int]):
        """insert(DocumentId, IndexedValue{field_length, terms}) (string_field.rs:155-177) with terms
        resolved to term ids; visible after commit()."""
        t = np.asarray(list(terms.keys()), np.uint32)
        f = np.asarray([min(v, 65535) for v in terms.values()], np.uint16)
        check(lib().oc_str_insert(self._h, field, int(doc_id), min(int(field_length), 65535), t.shape[0], _p(t), _p(f)))

    def commit(self):
        """compact(version) (string_field.rs:186-191)."""
        check(lib().oc_str_commit(self._h))

    def delete(self, doc_id):
        """One DocumentId or a sequence of them."""
        d = np.ascontiguousarray(np.atleast_1d(np.asarray(doc_id, np.uint64)).ravel())
        check(lib().oc_str_delete(self._h, _p(d), int(d.shape[0])))

    def info(self) -> dict:
        i = _lib.StrInfo()
        check(lib().oc_str_info(self._h, C.byref(i)))
        return {"total_documents": i.total_documents, "total_postings": i.total_postings,
                "unique_terms_count": i.unique_terms_count, "n_fields": i.n_fields, "device_bytes": i.device_bytes,
                "version": i.version, "pending_postings": i.pending_postings}

    def set_global(self, document_count: int, avg_field_len: Optional[Sequence[float]] = None):
        """This store is one shard: N of the idf and the per-field avg_field_len are corpus-wide values
        owned by the caller (kept across commits)."""
        a = None if avg_field_len is None else np.ascontiguousarray(avg_field_len, np.float32)
        check(lib().oc_str_set_global(self._h, int(document_count), _p(a)))


class DeviceFilter:
    """A FilterResult<DocumentId> evaluated to a bitmap that lives on the device (oc_filter_*): built once from
    the And / Or / Not tree of filters.py (filter.rs:344-392), reused by any number of searches."""

    def __init__(self, ctx: Context, handle, nbits: int):
        self.ctx, self._h, self.nbits = ctx, handle, int(nbits)

    @classmethod
    def from_ids(cls, ctx: Context, doc_ids, nbits: int) -> "DeviceFilter":
        ids = np.ascontiguousarray(np.asarray(list(doc_ids) if not isinstance(doc_ids, np.ndarray) else doc_ids, np.uint64))
        h = C.c_void_p()
        check(lib().oc_filter_from_ids(ctx._h, _p(ids), ids.shape[0], int(nbits), C.byref(h)))
        return cls(ctx, h, nbits)

    @classmethod
    def from_bits(cls, ctx: Context, bits: np.ndarray, nbits: int) -> "DeviceFilter":
        b = np.ascontiguousarray(bits, np.uint64)
        h = C.c_void_p()
        check(lib().oc_filter_from_bits(ctx._h, _p(b), int(nbits), C.byref(h)))
        return cls(ctx, h, nbits)

    @classmethod
    def from_expr(cls, ctx: Context, expr, nbits: int) -> "DeviceFilter":
        """filters.Ids / And / Or / Not tree -> device bitmap (leaves uploaded as id lists, combined on the device)."""
        from . import filters as F
        if isinstance(expr, F.Ids):
            return cls.from_ids(ctx, expr.doc_ids, nbits)
        if isinstance(expr, F.Not):
            a = cls.from_expr(ctx, expr.a, nbits)
            try:
                return ~a
            finally:
                a.close()
        if isinstance(expr, (F.And, F.Or)):
            a, b = cls.from_expr(ctx, expr.a, nbits), cls.from_expr(ctx, expr.b, nbits)
            try:
                return (a & b) if isinstance(expr, F.And) else (a | b)
            finally:
                a.close(); b.close()
        raise TypeError(f"not a filter expression: {expr!r}")

    def _bin(self, fn, other):
        h = C.c_void_p()
        check(fn(self._h, other._h, C.byref(h)))
        return DeviceFilter(self.ctx, h, self.nbits)

    def __and__(self, o): return self._bin(lib().oc_filter_and, o)
    def __or__(self, o): return self._bin(lib().oc_filter_or, o)

    def __invert__(self):
        h = C.c_void_p()
        check(lib().oc_filter_not(self._h, C.byref(h)))
        return DeviceFilter(self.ctx, h, self.nbits)

    def count(self) -> int:
        out = C.c_uint64()
        check(lib().oc_filter_count(self._h, C.byref(out)))
        return int(out.value)

    def read(self) -> np.ndarray:
        bits = np.zeros((self.nbits + 63) // 64, np.uint64)
        check(lib().oc_filter_read(self._h, _p(bits)))
        return bits

    def close(self):
        if self._h:
            lib().oc_filter_destroy(self._h)
            self._h = None


class FacetStore:
    """The filter fields of one Index laid out for facet counting on the device (oc_facets_*): per field the
    variants' document lists — bool true/false (bool_field.rs:182-208), string_filter keys
    (string_filter_field.rs:175-193), number fields sorted by value so a range is a slice (number_field.rs:368-387)."""

    def __init__(self, ctx: Context, nbits: int):
        self.ctx, self.nbits = ctx, int(nbits)
        self._h = C.c_void_p()
        check(lib().oc_facets_create(ctx._h, self.nbits, C.byref(self._h)))
        self.fields: Dict[str, dict] = {}

    def add_bool_field(self, name: str, true_docs, false_docs):
        return self._add_variants(name, "bool", {"true": true_docs, "false": false_docs})

    def add_string_field(self, name: str, docs_by_key: Dict[str, Sequence[int]]):
        return self._add_variants(name, "string", docs_by_key)

    def _add_variants(self, name, kind, docs_by_key):
        keys = list(docs_by_key)
        lists = [np.sort(np.asarray(list(docs_by_key[k]), np.uint64)) for k in keys]
        offs = np.zeros(len(keys) + 1, np.uint64)
        offs[1:] = np.cumsum([l.shape[0] for l in lists])
        docs = np.ascontiguousarray(np.concatenate(lists) if lists else np.zeros(0, np.uint64))
        fid = C.c_uint32()
        check(lib().oc_facets_add_field(self._h, len(keys), _p(offs), _p(docs), C.byref(fid)))
        self.fields[name] = {"id": fid.value, "kind": kind, "keys": keys}
        return fid.value

    def add_number_field(self, name: str, doc_ids, values):
        v = np.asarray(values, np.float64)
        d = np.asarray(doc_ids, np.uint64)
        o = np.argsort(v, kind="stable")
        v, d = np.ascontiguousarray(v[o]), np.ascontiguousarray(d[o])
        fid = C.c_uint32()
        check(lib().oc_facets_add_number_field(self._h, v.shape[0], _p(v), _p(d), C.byref(fid)))
        self.fields[name] = {"id": fid.value, "kind": "number"}
        return fid.value

    def close(self):
        if self._h:
            lib().oc_facets_destroy(self._h)
            self._h = None


def _number_label(x) -> str:
    return str(int(x)) if float(x) == int(x) else repr(float(x))


def search_facets(tsc: "TokenScoreContext", store: FacetStore, params: "TokenScoreParams", facets: Dict[str, dict], texts=None,
                  q_vecs: Optional[np.ndarray] = None) -> List[Dict[str, dict]]:
    """`facets` as in the reference's SearchParams: {"field": {"true": bool, "false": bool}} for a bool field,
    {"field": {"ranges": [{"from": a, "to": b}, ...]}} for a number field, {"field": {}} for a string_filter field.
    Returns, per query, {field: {"count": n_values, "values": {label: count}}} (FacetResult, types.rs:1508-1511;
    number labels "from-to", number_field.rs:382).  The where-filter of `params` is ignored, as in search.rs:361-396."""
    reqs, labels = [], []
    for name, d in facets.items():
        f = store.fields[name]
        if f["kind"] == "number":
            for r in d["ranges"]:
                reqs.append((f["id"], 0, float(r["from"]), float(r["to"])))
                labels.append((name, f"{_number_label(r['from'])}-{_number_label(r['to'])}"))
        else:
            for vi, key in enumerate(f["keys"]):
                if f["kind"] == "bool" and not d.get(key, False):
                    continue
                reqs.append((f["id"], vi, 0.0, 0.0))
                labels.append((name, key))
    sp, keep, B = tsc._build_params(params, texts, q_vecs)
    arr = (_lib.FacetReq * len(reqs))(*[_lib.FacetReq(*r) for r in reqs])
    out = np.zeros((B, max(len(reqs), 1)), np.uint64)
    check(lib().oc_search_facets(tsc.ctx._h, tsc.emb._h if tsc.emb else None, tsc.str._h if tsc.str else None, store._h,
                                 C.byref(sp), arr, len(reqs), _p(out)))
    res = []
    for q in range(B):
        r: Dict[str, dict] = {}
        for j, (name, label) in enumerate(labels):
            r.setdefault(name, {"count": 0, "values": {}})["values"][label] = int(out[q, j])
        for v in r.values():
            v["count"] = len(v["values"])
        res.append(r)
    return res


class SortStore:
    """The bool / number / date fields of one Index laid out for sortBy on the device (oc_sort_*): per field a dense
    rank of every document's value and the two walk orders of IndexSortContext::execute (read/index/sort.rs:186-264).
    Immutable once built: to refresh it, build a new one."""

    def __init__(self, ctx: Context, nbits: int):
        self.ctx, self.nbits = ctx, int(nbits)
        self._h = C.c_void_p()
        check(lib().oc_sort_create(ctx._h, self.nbits, C.byref(self._h)))
        self.fields: Dict[str, int] = {}

    def _add(self, name: str, fn, *args) -> int:
        fid = C.c_uint32()
        check(fn(self._h, *args, C.byref(fid)))
        self.fields[name] = fid.value
        return fid.value

    def add_number_field(self, name: str, doc_ids, values) -> int:
        """One number per document (i64 and f64 values compare as f64, number_field.rs:466-549); NaN is rejected."""
        d = np.ascontiguousarray(doc_ids, np.uint64)
        v = np.ascontiguousarray(values, np.float64)
        assert d.shape == v.shape
        return self._add(name, lib().oc_sort_add_number_field, d.shape[0], _p(d), _p(v))

    def add_date_field(self, name: str, doc_ids, timestamps) -> int:
        """One i64 timestamp per document, compared exactly (date_field.rs:239-246)."""
        d = np.ascontiguousarray(doc_ids, np.uint64)
        t = np.ascontiguousarray(timestamps, np.int64)
        assert d.shape == t.shape
        return self._add(name, lib().oc_sort_add_date_field, d.shape[0], _p(d), _p(t))

    def add_bool_field(self, name: str, true_docs, false_docs) -> int:
        """false before true ascending (index/sort.rs:210-241)."""
        t = np.ascontiguousarray(true_docs, np.uint64)
        f = np.ascontiguousarray(false_docs, np.uint64)
        return self._add(name, lib().oc_sort_add_bool_field, t.shape[0], _p(t), f.shape[0], _p(f))

    def close(self):
        if self._h:
            lib().oc_sort_destroy(self._h)
            self._h = None


def _sort_order(sort_by: dict) -> bool:
    """SortBy {property, order}: order defaults to ASC (types.rs:1351-1364); returns descending."""
    order = sort_by.get("order", "ASC")
    if order not in ("ASC", "DESC"):
        raise ValueError(f"sortBy order must be ASC or DESC, got {order!r}")
    return order == "DESC"


def search_sorted(tsc: "TokenScoreContext", store: SortStore, params: "TokenScoreParams", sort_by: dict, texts=None,
                  q_vecs: Optional[np.ndarray] = None, with_keys: bool = False):
    """sort_token_scores with Some(sort_by) (read/sort.rs:17-98): per query the score map's keys in the order of
    sort_by["property"], skip(offset).take(limit), each with its score-map value; count as execute_batch.  An unknown
    property raises KeyError (SortFieldNotFound).  with_keys: also return, per query, the sort value of each hit."""
    prop = sort_by["property"]
    if prop not in store.fields:
        raise KeyError(f"sort field not found: {prop!r}")
    desc = _sort_order(sort_by)
    sp, keep, B = tsc._build_params(params, texts, q_vecs)
    L = params.limit_hint
    docs, scores = np.empty((B, L), np.uint64), np.empty((B, L), np.float32)
    n, cnt, keys = np.empty(B, np.uint32), np.empty(B, np.uint64), np.empty((B, L), np.float64)
    check(lib().oc_search_sorted(tsc.ctx._h, tsc.emb._h if tsc.emb else None, tsc.str._h if tsc.str else None, store._h,
                                 store.fields[prop], int(desc), C.byref(sp), _p(docs), _p(scores), _p(n), _p(cnt), _p(keys)))
    hits = [SearchHits(docs[i, :n[i]].copy(), scores[i, :n[i]].copy(), int(cnt[i])) for i in range(B)]
    if with_keys:
        return hits, [keys[i, :n[i]].copy() for i in range(B)]
    return hits


def sort_last_forms(ctx: Context, n_queries: int) -> np.ndarray:
    """The selection form (0 = walk, 1 = gather) each query of the last search_sorted on ctx took."""
    out = np.zeros(max(n_queries, 1), np.uint8)
    check(lib().oc_sort_last_forms(ctx._h, int(n_queries), _p(out)))
    return out[:n_queries]


def merge_sorted_index_results(per_index, limit: int, offset: int = 0, order: str = "ASC") -> List[SearchHits]:
    """The multi-index union in field order (MergeSortedIterator, read/sort.rs:491-560) + skip/take: per_index = one
    (hits, keys) pair per index as search_sorted(..., with_keys=True) returns it, each run with
    limit_hint = limit+offset, offset = 0, vector_limit = limit.  count = the sum of the per-index counts."""
    k = len(per_index)
    B = len(per_index[0][0])
    stride = max(1, max(len(h.doc_ids) for hits, _ in per_index for h in hits))
    keep = []
    for hits, keys in per_index:
        d, s_, kk = np.zeros((B, stride), np.uint64), np.zeros((B, stride), np.float32), np.zeros((B, stride), np.float64)
        n, c = np.zeros(B, np.uint32), np.zeros(B, np.uint64)
        for q, h in enumerate(hits):
            m = len(h.doc_ids)
            d[q, :m], s_[q, :m], kk[q, :m], n[q], c[q] = h.doc_ids, h.scores, keys[q], m, h.count
        keep.append([d, s_, kk, n, c])
    arr = lambda j: (C.c_void_p * k)(*[r[j].ctypes.data for r in keep])
    od, os_ = np.zeros((B, limit), np.uint64), np.zeros((B, limit), np.float32)
    on, oc = np.zeros(B, np.uint32), np.zeros(B, np.uint64)
    check(lib().oc_merge_sorted_results(k, B, limit, offset, stride, int(_sort_order({"order": order})), arr(0), arr(1), arr(2),
                                        arr(3), arr(4), _p(od), _p(os_), _p(on), _p(oc)))
    return [SearchHits(od[i, :on[i]].copy(), os_[i, :on[i]].copy(), int(oc[i])) for i in range(B)]


def merge_index_results(per_index, limit: int, offset: int = 0) -> List[SearchHits]:
    """search_on_indexes' union of the per-index score maps + top_n + skip/take (search.rs:304-338, 482-498):
    per_index = one (doc_ids [B, limit+offset], scores, n, count) tuple per index, each obtained with
    limit' = limit+offset, offset' = 0, vector_limit = limit."""
    k = len(per_index)
    B, stride = per_index[0][0].shape
    keep = [[np.ascontiguousarray(a) for a in r] for r in per_index]
    arr = lambda j: (C.c_void_p * k)(*[r[j].ctypes.data for r in keep])
    od, os_ = np.zeros((B, limit), np.uint64), np.zeros((B, limit), np.float32)
    on, oc = np.zeros(B, np.uint32), np.zeros(B, np.uint64)
    check(lib().oc_merge_results(k, B, limit, offset, stride, arr(0), arr(1), arr(2), arr(3), _p(od), _p(os_), _p(on), _p(oc)))
    return [SearchHits(od[i, :on[i]].copy(), os_[i, :on[i]].copy(), int(oc[i])) for i in range(B)]


class TermDictionary:
    """Native term dictionaries of the string fields of one Index + batch query resolution (oc_dict_*,
    csrc/dict.h): tokenize (+ stem hook), then per field exact / prefix / Levenshtein expansion — what
    TextParser::tokenize_and_stem and the FST inside StringStorage do in the reference
    (token_score.rs:196-209, string_field.rs:208-225).  Host only: works without a GPU."""

    def __init__(self, n_fields: int = 1):
        self.n_fields = n_fields
        self._h = C.c_void_p()
        check(lib().oc_dict_create(n_fields, C.byref(self._h)))
        self._stem_cb = None

    def close(self):
        if self._h:
            lib().oc_dict_destroy(self._h)
            self._h = C.c_void_p()

    def add_terms(self, field: int, terms: Sequence[str]) -> np.ndarray:
        """Returns the (stable) ids of the terms; known terms keep their id, new ones get the next."""
        arr = (C.c_char_p * len(terms))(*[t.encode("utf-8") for t in terms])
        ids = np.zeros(len(terms), np.uint32)
        check(lib().oc_dict_add_terms(self._h, field, arr, len(terms), _p(ids)))
        return ids

    def lookup(self, field: int, term: str) -> Optional[int]:
        out = C.c_uint32()
        check(lib().oc_dict_lookup(self._h, field, term.encode("utf-8"), C.byref(out)))
        return None if out.value == 0xffffffff else int(out.value)

    def size(self, field: int) -> int:
        return int(lib().oc_dict_size(self._h, field))

    def set_stemmer(self, fn):
        """fn(token: str) -> Optional[str]; None / "" = no stem (test hook: a production binding passes a C function)."""
        def cb(tok, n, out, cap, _user):
            s = fn(C.string_at(tok, n).decode("utf-8"))
            if not s:
                return 0
            b = s.encode("utf-8")
            if len(b) > cap:
                return 0
            C.memmove(out, b, len(b))
            return len(b)
        self._stem_cb = _lib.STEM_FN(cb) if fn is not None else None
        check(lib().oc_dict_set_stemmer(self._h, C.cast(self._stem_cb, C.c_void_p) if fn is not None else None, None))

    def use_english_stemmer(self):
        """Install the built-in Snowball English (Porter2) stemmer (oc_stem_english)."""
        check(lib().oc_dict_set_stemmer(self._h, C.cast(lib().oc_stem_english, C.c_void_p), None))

    @staticmethod
    def stem_english(token: str) -> str:
        b = token.encode("utf-8")
        out = C.create_string_buffer(len(b) + 8)
        n = lib().oc_stem_english(b, len(b), out, len(b) + 8, None)
        return out.raw[:n].decode("utf-8") if n else token

    def resolve_batch(self, texts: Sequence[str], exact: bool = False, tolerance: Optional[int] = None,
                      boost: Optional[Sequence[float]] = None, properties: Optional[Sequence[int]] = None,
                      exact_match_boost: float = 0.0) -> "TextQueryBatch":
        """SearchParams{tokens, exact_match, boost, tolerance} for B queries at once (token_score.rs:235-242)
        -> the packed CSR arrays oc_search takes."""
        rp = _lib.ResolveParams()
        arr = (C.c_char_p * len(texts))(*[t.encode("utf-8") for t in texts])
        rp.texts, rp.n_queries = arr, len(texts)
        rp.exact, rp.tolerance = int(bool(exact)), -1 if tolerance is None else int(tolerance)
        fb = None if boost is None else np.ascontiguousarray(boost, np.float32)
        fm = None
        if properties is not None:
            fm = np.zeros(self.n_fields, np.uint8)
            fm[list(properties)] = 1
        rp.field_boost, rp.field_mask, rp.exact_match_boost = _p(fb), _p(fm), float(exact_match_boost)
        res = C.c_void_p()
        check(lib().oc_dict_resolve(self._h, C.byref(rp), C.byref(res)))
        try:
            ptrs = [C.c_void_p() for _ in range(5)]
            nt, ne = C.c_uint32(), C.c_uint32()
            lib().oc_resolved_arrays(res, *[C.byref(x) for x in ptrs], C.byref(nt), C.byref(ne))
            B = len(texts)

            def arr_of(ptr, n, ct, dt):
                return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), shape=(max(n, 1),))[:n].astype(dt, copy=True)
            out = TextQueryBatch.__new__(TextQueryBatch)
            out.n_queries = B
            out.q_token_offsets = arr_of(ptrs[0], B + 1, C.c_uint32, np.uint32)
            out.token_term_offsets = arr_of(ptrs[1], nt.value + 1, C.c_uint32, np.uint32)
            out.term_field = arr_of(ptrs[2], ne.value, C.c_uint32, np.uint32)
            out.term_id = arr_of(ptrs[3], ne.value, C.c_uint32, np.uint32)
            out.term_weight = arr_of(ptrs[4], ne.value, C.c_float, np.float32)
            return out
        finally:
            lib().oc_resolved_free(res)


class TextQueryBatch:
    """B resolved queries packed as the CSR arrays oc_search takes (q -> tokens -> expanded terms)."""

    def query(self, i: int) -> TextQuery:
        """The i-th query as a TextQuery (tests: compare with a host-side resolution)."""
        t0, t1 = int(self.q_token_offsets[i]), int(self.q_token_offsets[i + 1])
        e0, e1 = int(self.token_term_offsets[t0]), int(self.token_term_offsets[t1])
        return TextQuery((self.token_term_offsets[t0:t1 + 1] - np.uint32(e0)).astype(np.uint32), self.term_field[e0:e1].copy(),
                         self.term_id[e0:e1].copy(), self.term_weight[e0:e1].copy())

    def __init__(self, texts: Sequence[TextQuery]):
        B = len(texts)
        self.n_queries = B
        qoff = np.zeros(B + 1, np.uint32)
        tto, tf_, tid, tw = [np.zeros(1, np.uint32)], [], [], []
        ntok = nterm = 0
        for i, t in enumerate(texts):
            ntok += t.n_tokens
            qoff[i + 1] = ntok
            tto.append(t.token_term_offsets[1:].astype(np.uint32) + np.uint32(nterm))
            nterm += int(t.token_term_offsets[-1])
            tf_.append(t.term_field); tid.append(t.term_id); tw.append(t.term_weight)
        self.q_token_offsets = qoff
        self.token_term_offsets = np.ascontiguousarray(np.concatenate(tto), np.uint32)
        self.term_field = np.ascontiguousarray(np.concatenate(tf_) if tf_ else np.zeros(0), np.uint32)
        self.term_id = np.ascontiguousarray(np.concatenate(tid) if tid else np.zeros(0), np.uint32)
        self.term_weight = np.ascontiguousarray(np.concatenate(tw) if tw else np.zeros(0), np.float32)


@dataclass
class TokenScoreParams:
    """token_score.rs:31-41 (mode already resolved; boost/properties are folded into the
    resolved TextQuery by the host-side term resolution)."""
    mode: int
    limit_hint: int = 10
    offset: int = 0
    similarity: float = 0.7          # types.rs:881-885
    threshold: Optional[float] = None
    filtered_doc_ids: Optional[np.ndarray] = None
    filter_nbits: int = 0
    device_filter: Optional["DeviceFilter"] = None   # device-resident bitmap (oc_filter_*); wins over filtered_doc_ids
    vector_limit: int = 0            # 0 => limit_hint (search.rs:330-336); see oc_search_params.vector_limit
    omc_doc_ids: Optional[np.ndarray] = None   # ascending
    omc_mult: Optional[np.ndarray] = None
    sharded: bool = False
    shard_tombstones: bool = False   # OC_SHARD_TOMBSTONES: some rank's string store holds uncommitted deletes
    shard_count_df: bool = False     # OC_SHARD_COUNT_DF: some rank's store lacks the corpus-wide df tables


class TokenScoreContext:
    """token_score.rs:49-57 + execute :460-509, fused with OMC, count and top-N.

    execute_batch() is the GPU drop-in: it returns, per query, the top (limit) hits after
    offset and the total match count — what search_on_indexes derives from the score map
    (search.rs:482-498) — instead of materialising the whole HashMap on the host."""

    def __init__(self, ctx: Context, embedding_field: Optional[EmbeddingFieldStorage],
                 string_fields: Optional[StringFieldStorage]):
        self.ctx, self.emb, self.str = ctx, embedding_field, string_fields

    def execute_batch(self, params: TokenScoreParams, texts=None,
                      q_vecs: Optional[np.ndarray] = None) -> List[SearchHits]:
        docs, scores, n, cnt = self.execute_batch_arrays(params, texts, q_vecs)
        return [SearchHits(docs[i, :n[i]].copy(), scores[i, :n[i]].copy(), int(cnt[i])) for i in range(docs.shape[0])]

    def execute_batch_arrays(self, params: TokenScoreParams, texts=None, q_vecs: Optional[np.ndarray] = None):
        """Same call, results as arrays: (doc_ids [B,limit], scores [B,limit], n [B], count [B]).
        `texts` is a sequence of TextQuery or a pre-packed TextQueryBatch (term resolution happens
        before the hot path in the reference as well: token_score.rs:196-209)."""
        sp, keep, B = self._build_params(params, texts, q_vecs)
        docs = np.empty((B, params.limit_hint), np.uint64)
        scores = np.empty((B, params.limit_hint), np.float32)
        n = np.empty(B, np.uint32)
        cnt = np.empty(B, np.uint64)
        check(lib().oc_search(self.ctx._h, self.emb._h if self.emb else None, self.str._h if self.str else None,
                              C.byref(sp), _p(docs), _p(scores), _p(n), _p(cnt)))
        return docs, scores, n, cnt

    def _build_params(self, params: TokenScoreParams, texts=None, q_vecs: Optional[np.ndarray] = None):
        """oc_search_params for a batch; `keep` holds the arrays the struct points into."""
        if texts is not None and not isinstance(texts, TextQueryBatch):
            texts = TextQueryBatch(texts)
        B = texts.n_queries if texts is not None else int(np.asarray(q_vecs).reshape(-1, self.emb.dim).shape[0])
        sp = SearchParams()
        sp.mode = params.mode
        sp.n_queries = B
        sp.limit, sp.offset = params.limit_hint, params.offset
        sp.similarity = params.similarity
        sp.threshold = -1.0 if params.threshold is None else params.threshold
        sp.bm25_k, sp.bm25_b = BM25_K, BM25_B
        keep = []
        if params.mode in (MODE_VECTOR, MODE_HYBRID):
            qv = np.ascontiguousarray(q_vecs, np.float32).reshape(B, self.emb.dim)
            keep.append(qv)
            sp.q_vecs = _p(qv)
        if params.mode in (MODE_FULLTEXT, MODE_HYBRID):
            keep.append(texts)
            sp.q_token_offsets, sp.token_term_offsets = _p(texts.q_token_offsets), _p(texts.token_term_offsets)
            sp.term_field, sp.term_id, sp.term_weight = _p(texts.term_field), _p(texts.term_id), _p(texts.term_weight)
        sp.vector_limit = int(params.vector_limit)
        if params.device_filter is not None:
            keep.append(params.device_filter)
            sp.filter = params.device_filter._h
        elif params.filtered_doc_ids is not None:
            fb = np.ascontiguousarray(params.filtered_doc_ids, np.uint64)
            keep.append(fb)
            sp.filter_bits, sp.filter_nbits = _p(fb), int(params.filter_nbits)
        if params.omc_doc_ids is not None and len(params.omc_doc_ids):
            od = np.ascontiguousarray(params.omc_doc_ids, np.uint64)
            om = np.ascontiguousarray(params.omc_mult, np.float32)
            keep += [od, om]
            sp.omc_doc_ids, sp.omc_mult, sp.n_omc = _p(od), _p(om), od.shape[0]
        sp.sharded = (1 | (2 if params.shard_tombstones else 0) | (4 if params.shard_count_df else 0)) if params.sharded else 0
        return sp, keep, B

    def execute(self, params: TokenScoreParams, results: Dict[int, float], text: Optional[TextQuery] = None,
                q_vec: Optional[np.ndarray] = None) -> int:
        """Reference-shaped call: `results.extend(scores)` for one query; returns the match count.
        limit and offset are passed through unchanged (the vector stage's candidate depth is limit_hint =
        limit, NOT limit + offset: search.rs:330-336), so `results` receives the rows [offset, offset+limit)
        of the ranking — the rest of the score map never leaves the GPU."""
        hits = self.execute_batch(params, None if text is None else [text], q_vec)[0]
        for d, s in zip(hits.doc_ids, hits.scores):
            results[int(d)] = np.float32(s)
        return hits.count


class SearchBatcher:
    """Micro-batching front (oc_batcher_*, csrc/batcher.h): many threads call search() with ONE query
    each — the way the reference's request tasks call TokenScoreContext::execute — and the library
    coalesces concurrent calls that share (mode, limit, offset, similarity, threshold) into one
    batched oc_search.  ctypes releases the GIL while a caller is blocked in the library."""

    def __init__(self, tsc: TokenScoreContext, max_batch: int = 256, max_wait_us: int = 200):
        self.tsc = tsc
        h = C.c_void_p()
        check(lib().oc_batcher_create(tsc.ctx._h, tsc.emb._h if tsc.emb else None, tsc.str._h if tsc.str else None,
                                      int(max_batch), int(max_wait_us), C.byref(h)))
        self._h = h

    def search(self, params: TokenScoreParams, text: Optional[TextQuery] = None,
               q_vec: Optional[np.ndarray] = None) -> SearchHits:
        sp, keep, B = self.tsc._build_params(params, None if text is None else [text],
                                             None if q_vec is None else np.asarray(q_vec, np.float32).reshape(1, -1))
        assert B == 1
        L = params.limit_hint
        docs, scores = np.empty(L, np.uint64), np.empty(L, np.float32)
        n, cnt = np.zeros(1, np.uint32), np.zeros(1, np.uint64)
        check(lib().oc_batcher_search(self._h, C.byref(sp), _p(docs), _p(scores), _p(n), _p(cnt)))
        k = int(n[0])
        return SearchHits(docs[:k].copy(), scores[:k].copy(), int(cnt[0]))

    def stats(self) -> dict:
        q, b, d = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(lib().oc_batcher_stats(self._h, C.byref(q), C.byref(b), C.byref(d)))
        return {"queries": q.value, "batches": b.value, "direct": d.value}

    def close(self):
        if self._h:
            lib().oc_batcher_destroy(self._h)
            self._h = None


def search(ctx: Context, emb: Optional[EmbeddingFieldStorage], strs: Optional[StringFieldStorage], mode: str,
           texts: Optional[Sequence[TextQuery]] = None, q_vecs: Optional[np.ndarray] = None, limit: int = 10,
           offset: int = 0, similarity: float = 0.7, threshold: Optional[float] = None, **kw) -> List[SearchHits]:
    """search() surface of the hot path: mode = "fulltext" | "vector" | "hybrid" (types.rs:924-999;
    "default" == fulltext)."""
    m = {"fulltext": MODE_FULLTEXT, "default": MODE_FULLTEXT, "vector": MODE_VECTOR, "hybrid": MODE_HYBRID}[mode]
    p = TokenScoreParams(mode=m, limit_hint=limit, offset=offset, similarity=similarity, threshold=threshold, **kw)
    return TokenScoreContext(ctx, emb, strs).execute_batch(p, texts, q_vecs)
