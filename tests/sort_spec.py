"""numpy statement of sortBy (read/sort.rs:48-98 sort_token_scores_by_field, :236-257 truncate) and of the two device
selection forms of K6 (csrc/sort.cuh), shared by the host and GPU tests.

A field is (doc_ids, values): one value per document.  The walk visits the value groups in the requested order
(IndexSortContext::execute, read/index/sort.rs:186-264), ascending DocumentId inside a group, and emits a document
when it is a key of the score map; documents without a value are never emitted."""
import numpy as np


def field_order(doc_ids, values, descending):
    """DocumentIds in walk order: value ascending / descending, DocumentId ascending inside equal values."""
    d = np.asarray(doc_ids, np.uint64)
    _, r = np.unique(np.asarray(values), return_inverse=True)   # exact order for f64, i64 and bool values
    r = r.astype(np.int64)
    return d[np.lexsort((d, -r if descending else r))]


def sort_by_field(map_docs, map_scores, doc_ids, values, top_count, descending):
    """sort_token_scores_by_field + truncate: the first top_count map keys in walk order, with their map values."""
    score = dict(zip(np.asarray(map_docs, np.uint64).tolist(), np.asarray(map_scores, np.float32).tolist()))
    out_d, out_s = [], []
    for d in field_order(doc_ids, values, descending).tolist():
        if len(out_d) >= top_count:
            break
        if d in score:
            out_d.append(d); out_s.append(score[d])
    return np.asarray(out_d, np.uint64), np.asarray(out_s, np.float32)


def dense_rank(doc_ids, values, nbits):
    """rank[nbits]: dense rank of each document's value (ties share a rank), -1 = no value."""
    v = np.asarray(values)
    uniq, inv = np.unique(v, return_inverse=True)
    rank = np.full(nbits, -1, np.int64)
    rank[np.asarray(doc_ids, np.int64)] = inv
    return rank, len(uniq)


def select_walk(bits, order, n_keep):
    """Walk form: stream the order permutation, keep the first n_keep documents set in the bitmap."""
    hit = bits[order.astype(np.int64)] if order.size else np.zeros(0, bool)
    return order[hit][:n_keep]


def select_gather(bits, rank, n_ranks, n_keep, descending):
    """Gather form: keys (rank' << 32 | id) of the set documents that have a value, the n_keep smallest ascending."""
    docs = np.flatnonzero(bits[: rank.shape[0]])
    docs = docs[rank[docs] >= 0]
    r = rank[docs]
    if descending:
        r = n_ranks - 1 - r
    keys = (r.astype(np.uint64) << np.uint64(32)) | docs.astype(np.uint64)
    return (np.sort(keys)[:n_keep] & np.uint64(0xFFFFFFFF)).astype(np.uint64)


def merge_sorted(per_index, limit, offset, descending):
    """MergeSortedIterator over per-index (doc_ids, scores, keys, count) lists already in field order: the head with the
    first key wins, equal keys go to the lower index; then skip(offset).take(limit); count = sum of counts."""
    rows = []
    for i, (d, s, k, _) in enumerate(per_index):
        for j in range(len(d)):
            rows.append(((-k[j] if descending else k[j]), i, j, int(d[j]), np.float32(s[j])))
    rows.sort(key=lambda r: (r[0], r[1], r[2]))
    rows = rows[offset:offset + limit]
    return (np.asarray([r[3] for r in rows], np.uint64), np.asarray([r[4] for r in rows], np.float32),
            sum(int(c) for *_, c in per_index))
