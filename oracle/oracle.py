"""ctypes wrapper over oracle/liboracle.so — the CPU restatement of the reference's search path.

TEST INFRASTRUCTURE ONLY (see oracle.h): imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference leg.  Never imported by oramacore_b200/.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle.so")


def build(force: bool = False) -> str:
    src = [os.path.join(_HERE, "oracle.c"), os.path.join(_HERE, "oracle.h")]
    stale = (not os.path.exists(_SO)) or any(
        os.path.exists(s) and os.path.getmtime(s) > os.path.getmtime(_SO) for s in src)
    if force or stale:
        if not os.path.exists(src[0]):
            raise RuntimeError("oracle sources missing")
        subprocess.check_call(["make", "-C", _HERE, "-B", "liboracle.so"], stdout=subprocess.DEVNULL)
    return _SO


class _Field(C.Structure):
    _fields_ = [("avg_field_len", C.c_float), ("n_terms", C.c_uint32),
                ("term_offsets", C.c_void_p), ("post_row", C.c_void_p),
                ("post_tf", C.c_void_p), ("post_len", C.c_void_p), ("global_df", C.c_void_p)]


class _StrIndex(C.Structure):
    _fields_ = [("n_fields", C.c_uint32), ("fields", C.POINTER(_Field)), ("n_rows", C.c_uint64),
                ("row_doc_ids", C.c_void_p), ("document_count", C.c_uint64)]


class _TextQuery(C.Structure):
    _fields_ = [("n_tokens", C.c_uint32), ("token_term_offsets", C.c_void_p),
                ("term_field", C.c_void_p), ("term_id", C.c_void_p), ("term_weight", C.c_void_p)]


class _TextParams(C.Structure):
    _fields_ = [("b", C.c_float), ("k", C.c_float), ("threshold", C.c_float),
                ("filter_bits", C.c_void_p), ("filter_nbits", C.c_uint64)]


class _Map(C.Structure):
    _fields_ = [("doc", C.POINTER(C.c_uint64)), ("score", C.POINTER(C.c_float)),
                ("n", C.c_size_t), ("cap", C.c_size_t)]


class _EmbStore(C.Structure):
    _fields_ = [("dim", C.c_uint32), ("n_rows", C.c_uint64), ("rows", C.c_void_p),
                ("row_doc_ids", C.c_void_p), ("deleted", C.c_void_p), ("is_e5", C.c_int),
                ("row_norms", C.c_void_p)]


class _SearchReq(C.Structure):
    _fields_ = [("mode", C.c_int), ("limit", C.c_uint32), ("offset", C.c_uint32),
                ("similarity", C.c_float), ("q_vec", C.c_void_p),
                ("text", C.POINTER(_TextQuery)), ("tp", C.POINTER(_TextParams)),
                ("omc_doc", C.c_void_p), ("omc_mult", C.c_void_p), ("n_omc", C.c_size_t)]


_lib = None


def lib():
    """Loads the library build() made without recompiling it, so callers such as bench.py never write
    into the tree; it is compiled here only when it is missing."""
    global _lib
    if _lib is None:
        L = C.CDLL(_SO if os.path.exists(_SO) else build())
        L.orc_idf.restype = C.c_float
        L.orc_idf.argtypes = [C.c_float, C.c_uint64]
        L.orc_normalized_tf.restype = C.c_float
        L.orc_normalized_tf.argtypes = [C.c_uint32, C.c_uint32, C.c_float, C.c_float]
        L.orc_bm25f_score.restype = C.c_float
        L.orc_bm25f_score.argtypes = [C.c_float, C.c_float, C.c_float]
        L.orc_bm25_legacy_add.restype = C.c_float
        L.orc_bm25_legacy_add.argtypes = [C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_uint64,
                                          C.c_float, C.c_float, C.c_float, C.c_float]
        L.orc_rescale_score.restype = C.c_float
        L.orc_rescale_score.argtypes = [C.c_float, C.c_int]
        L.orc_row_norms.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
        L.orc_row_norms.restype = None
        L.orc_map_free.argtypes = [C.POINTER(_Map)]
        L.orc_fulltext.argtypes = [C.POINTER(_StrIndex), C.POINTER(_TextQuery), C.POINTER(_TextParams), C.POINTER(_Map)]
        L.orc_vector.argtypes = [C.POINTER(_EmbStore), C.c_void_p, C.c_uint32, C.c_float, C.c_void_p, C.c_uint64, C.POINTER(_Map)]
        L.orc_vector_f64.argtypes = [C.POINTER(_EmbStore), C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
        L.orc_hybrid_combine.argtypes = [C.POINTER(_Map), C.POINTER(_Map), C.POINTER(_Map)]
        L.orc_apply_omc.argtypes = [C.POINTER(_Map), C.c_void_p, C.c_void_p, C.c_size_t]
        L.orc_top_n.restype = C.c_size_t
        L.orc_top_n.argtypes = [C.POINTER(_Map), C.c_size_t, C.c_void_p, C.c_void_p]
        L.orc_search.argtypes = [C.POINTER(_StrIndex), C.POINTER(_EmbStore), C.POINTER(_SearchReq),
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_search_batch.argtypes = [C.POINTER(_StrIndex), C.POINTER(_EmbStore), C.POINTER(_SearchReq),
                                       C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


# ---------------------------------------------------------------- scalar helpers
def idf(n_docs: float, df: int) -> float:
    return float(lib().orc_idf(n_docs, df))


def normalized_tf(tf: int, flen: int, avg: float, b: float = 0.75) -> float:
    return float(lib().orc_normalized_tf(tf, flen, avg, b))


def bm25f_score(S: float, k: float, idf_: float) -> float:
    return float(lib().orc_bm25f_score(S, k, idf_))


def bm25_legacy_add(tf, flen, avg, total_docs, df, k, weight, b, boost) -> float:
    return float(lib().orc_bm25_legacy_add(tf, flen, avg, total_docs, df, k, weight, b, boost))


def rescale_score(s: float, is_e5: bool) -> float:
    return float(lib().orc_rescale_score(s, int(is_e5)))


# ---------------------------------------------------------------- index / store views
class StrIndex:
    """Keeps numpy arrays alive behind an orc_str_index."""

    def __init__(self, data, global_df=None):  # data: oramacore_b200.types.StringIndexData (duck-typed)
        self._keep = []
        arr = (_Field * max(1, len(data.fields)))()
        for i, f in enumerate(data.fields):
            to = np.ascontiguousarray(f.term_offsets, np.uint64)
            pr = np.ascontiguousarray(f.post_row, np.uint32)
            pt = np.ascontiguousarray(f.post_tf, np.uint16)
            pl = np.ascontiguousarray(f.post_len, np.uint16)
            gd = None if global_df is None else np.ascontiguousarray(global_df[i], np.uint32)
            self._keep += [to, pr, pt, pl, gd]
            arr[i] = _Field(float(f.avg_field_len), to.shape[0] - 1, _p(to), _p(pr), _p(pt), _p(pl), _p(gd))
        self._fields = arr
        rd = None if data.row_doc_ids is None else np.ascontiguousarray(data.row_doc_ids, np.uint64)
        self._keep.append(rd)
        self.c = _StrIndex(len(data.fields), arr, int(data.n_rows), _p(rd), int(data.document_count))


class EmbStore:
    def __init__(self, rows: np.ndarray, row_doc_ids: Optional[np.ndarray] = None,
                 deleted: Optional[np.ndarray] = None, is_e5: bool = False):
        self.rows = np.ascontiguousarray(rows, np.float32)
        self.rd = None if row_doc_ids is None else np.ascontiguousarray(row_doc_ids, np.uint64)
        self.dl = None if deleted is None else np.ascontiguousarray(deleted, np.uint8)
        n, d = self.rows.shape
        self.norms = np.zeros(n, np.float32)  # cached |x| (what any real store precomputes)
        lib().orc_row_norms(_p(self.rows), n, d, _p(self.norms))
        self.c = _EmbStore(d, n, _p(self.rows), _p(self.rd), _p(self.dl), int(is_e5), _p(self.norms))


class _TQ:
    def __init__(self, q):  # q: TextQuery
        self.a = [np.ascontiguousarray(q.token_term_offsets, np.uint32),
                  np.ascontiguousarray(q.term_field, np.uint32),
                  np.ascontiguousarray(q.term_id, np.uint32),
                  np.ascontiguousarray(q.term_weight, np.float32)]
        self.c = _TextQuery(self.a[0].shape[0] - 1, _p(self.a[0]), _p(self.a[1]), _p(self.a[2]), _p(self.a[3]))


class _TP:
    def __init__(self, threshold=None, filter_bits=None, filter_nbits=0, b=0.75, k=1.2):
        self.fb = None if filter_bits is None else np.ascontiguousarray(filter_bits, np.uint64)
        self.c = _TextParams(b, k, -1.0 if threshold is None else float(threshold), _p(self.fb),
                             int(filter_nbits))


def _take_map(m: _Map):
    n = m.n
    d = np.ctypeslib.as_array(m.doc, shape=(max(n, 1),))[:n].copy() if n else np.zeros(0, np.uint64)
    s = np.ctypeslib.as_array(m.score, shape=(max(n, 1),))[:n].copy() if n else np.zeros(0, np.float32)
    lib().orc_map_free(C.byref(m))
    return d.astype(np.uint64), s.astype(np.float32)


def _mk_map(doc: np.ndarray, score: np.ndarray):
    d = np.ascontiguousarray(doc, np.uint64)
    s = np.ascontiguousarray(score, np.float32)
    m = _Map(d.ctypes.data_as(C.POINTER(C.c_uint64)), s.ctypes.data_as(C.POINTER(C.c_float)), d.shape[0], d.shape[0])
    return m, (d, s)


def make_filter_bits(allowed_doc_ids: Sequence[int], nbits: int) -> np.ndarray:
    bits = np.zeros((nbits + 63) // 64, np.uint64)
    ids = np.asarray(list(allowed_doc_ids), np.uint64)
    ids = ids[ids < nbits]
    np.bitwise_or.at(bits, (ids >> np.uint64(6)).astype(np.int64), np.uint64(1) << (ids & np.uint64(63)))
    return bits


# ---------------------------------------------------------------- the restated functions
def fulltext(ix: StrIndex, q, threshold=None, filter_bits=None, filter_nbits=0):
    """search_full_text: returns (doc_ids sorted, scores) = the whole score map."""
    tq, tp, m = _TQ(q), _TP(threshold, filter_bits, filter_nbits), _Map()
    rc = lib().orc_fulltext(C.byref(ix.c), C.byref(tq.c), C.byref(tp.c), C.byref(m))
    assert rc == 0
    return _take_map(m)


def vector(st: EmbStore, target: np.ndarray, limit: int, similarity: float,
           filter_bits=None, filter_nbits=0):
    t = np.ascontiguousarray(target, np.float32)
    fb = None if filter_bits is None else np.ascontiguousarray(filter_bits, np.uint64)
    m = _Map()
    rc = lib().orc_vector(C.byref(st.c), _p(t), limit, similarity, _p(fb), int(filter_nbits), C.byref(m))
    assert rc == 0
    return _take_map(m)


def vector_f64(st: EmbStore, target: np.ndarray, limit: int):
    t = np.ascontiguousarray(target, np.float32)
    od = np.zeros(limit, np.uint64)
    oc = np.zeros(limit, np.float64)
    n = lib().orc_vector_f64(C.byref(st.c), _p(t), limit, _p(od), _p(oc))
    assert n >= 0
    return od[:n], oc[:n]


def hybrid_combine(vec, ft):
    mv, k1 = _mk_map(*vec)
    mf, k2 = _mk_map(*ft)
    out = _Map()
    rc = lib().orc_hybrid_combine(C.byref(mv), C.byref(mf), C.byref(out))
    assert rc == 0
    return _take_map(out)


def apply_omc(scores, omc_doc, omc_mult):
    m, (d, s) = _mk_map(*scores)
    od = np.ascontiguousarray(omc_doc, np.uint64)
    om = np.ascontiguousarray(omc_mult, np.float32)
    lib().orc_apply_omc(C.byref(m), _p(od), _p(om), od.shape[0])
    return d, s


def top_n(scores, n: int):
    m, _k = _mk_map(*scores)
    od = np.zeros(max(n, 1), np.uint64)
    os_ = np.zeros(max(n, 1), np.float32)
    got = lib().orc_top_n(C.byref(m), n, _p(od), _p(os_))
    return od[:got], os_[:got]


class SearchBatch:
    """Builds an array of orc_search_req and runs orc_search / orc_search_batch."""

    def __init__(self, ix: Optional[StrIndex], st: Optional[EmbStore]):
        self.ix, self.st = ix, st
        self._keep: List = []
        self._reqs: List[_SearchReq] = []

    def add(self, mode: int, limit: int = 10, offset: int = 0, similarity: float = 0.7,
            q_vec: Optional[np.ndarray] = None, text=None, threshold=None,
            filter_bits=None, filter_nbits=0, omc_doc=None, omc_mult=None):
        tq = _TQ(text) if text is not None else None
        tp = _TP(threshold, filter_bits, filter_nbits)
        qv = None if q_vec is None else np.ascontiguousarray(q_vec, np.float32)
        od = None if omc_doc is None else np.ascontiguousarray(omc_doc, np.uint64)
        om = None if omc_mult is None else np.ascontiguousarray(omc_mult, np.float32)
        self._keep += [tq, tp, qv, od, om]
        r = _SearchReq(mode, limit, offset, similarity, _p(qv),
                       C.pointer(tq.c) if tq is not None else None, C.pointer(tp.c),
                       _p(od), _p(om), 0 if od is None else od.shape[0])
        self._reqs.append(r)

    def run(self, n_threads: int = 1):
        n = len(self._reqs)
        arr = (_SearchReq * n)(*self._reqs)
        stride = max(r.limit for r in self._reqs)
        od = np.zeros((n, stride), np.uint64)
        os_ = np.zeros((n, stride), np.float32)
        on = np.zeros(n, np.uint32)
        oc = np.zeros(n, np.uint64)
        rc = lib().orc_search_batch(C.byref(self.ix.c) if self.ix else None,
                                    C.byref(self.st.c) if self.st else None,
                                    arr, n, n_threads, _p(od), _p(os_), _p(on), _p(oc))
        assert rc == 0
        return od, os_, on, oc
