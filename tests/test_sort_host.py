"""sortBy without a device: the numpy statement of sort_token_scores_by_field + truncate, the two selection forms of K6
(walk and gather select the same documents), and oc_merge_sorted_results (host only) against MergeSortedIterator."""
import numpy as np
import pytest

import oramacore_b200 as ob
from oramacore_b200.types import SearchHits
from sort_spec import dense_rank, field_order, merge_sorted, select_gather, select_walk, sort_by_field


def test_statement_orders_groups_then_ascending_ids():
    # src/tests/sort.rs:418-493: three documents share the key; the where-filter leaves 1 and 3
    d, s = sort_by_field([1, 3], [0.5, 0.25], [1, 2, 3], [2.0, 2.0, 2.0], 10, False)
    assert d.tolist() == [1, 3] and s.tolist() == [0.5, 0.25]
    # bool: false before true ascending, true before false descending (index/sort.rs:210-241)
    assert field_order([1, 2], [False, True], False).tolist() == [1, 2]
    assert field_order([1, 2], [False, True], True).tolist() == [2, 1]
    # ties stay in ascending id in both orders; documents without a value are never emitted
    assert field_order([5, 3, 9, 1], [1.0, 2.0, 1.0, 2.0], True).tolist() == [1, 3, 5, 9]
    d, _ = sort_by_field([0, 1, 2, 3], [1, 1, 1, 1], [2, 3], [7, 8], 10, False)
    assert d.tolist() == [2, 3]


def _case(rng, nbits, kind):
    n_pop = int(nbits * 0.9)
    docs = rng.choice(nbits, size=n_pop, replace=False).astype(np.uint64)
    vals = rng.integers(0, 4, size=n_pop).astype(np.float64) if kind == "ties" else rng.normal(size=n_pop)
    if kind == "empty":
        bits = np.zeros(nbits, bool)
    elif kind == "all":
        bits = np.ones(nbits, bool)
    else:
        bits = rng.random(nbits) < (0.3 if kind == "ties" else 0.01)
    return docs, vals, bits


@pytest.mark.parametrize("kind", ["random", "ties", "empty", "all"])
@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("limit,offset", [(10, 0), (7, 5), (1000, 24)])
def test_walk_and_gather_select_the_same_documents(kind, descending, limit, offset):
    rng = np.random.default_rng(["random", "ties", "empty", "all"].index(kind) * 4096 + int(descending) * 2048 + limit)
    nbits = 5000
    docs, vals, bits = _case(rng, nbits, kind)
    n_keep = limit + offset
    rank, n_ranks = dense_rank(docs, vals, nbits)
    order = field_order(docs, vals, descending)
    walk = select_walk(bits, order, n_keep)
    gather = select_gather(bits, rank, n_ranks, n_keep, descending)
    assert walk.tolist() == gather.tolist()
    keys = np.flatnonzero(bits).astype(np.uint64)
    exp, _ = sort_by_field(keys, np.zeros(keys.shape[0], np.float32), docs, vals, n_keep, descending)
    assert walk.tolist() == exp.tolist()
    assert walk[offset:offset + limit].shape[0] == max(0, min(limit, exp.shape[0] - offset))


def _index_lists(rng, ids, descending, top):
    vals = rng.integers(0, 5, size=ids.shape[0]).astype(np.float64)    # heavy ties across indexes
    keys = ids[rng.random(ids.shape[0]) < 0.7]
    scores = rng.random(keys.shape[0]).astype(np.float32)
    d, s = sort_by_field(keys, scores, ids, vals, top, descending)
    k = dict(zip(ids.tolist(), vals.tolist()))
    return d, s, np.asarray([k[x] for x in d.tolist()], np.float64), keys.shape[0]


@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("limit,offset", [(5, 0), (6, 7), (40, 3)])
def test_merge_sorted_results_matches_merge_sorted_iterator(descending, limit, offset):
    rng = np.random.default_rng(7 + limit)
    B = 3
    all_ids = rng.permutation(300).astype(np.uint64)
    parts = [np.sort(all_ids[:100]), np.sort(all_ids[100:220]), np.sort(all_ids[220:])]
    per_index_q = [[_index_lists(rng, ids, descending, limit + offset) for _ in range(B)] for ids in parts]
    per_index = [([SearchHits(d, s, c) for d, s, _, c in rows], [k for _, _, k, _ in rows]) for rows in per_index_q]
    got = ob.merge_sorted_index_results(per_index, limit, offset, "DESC" if descending else "ASC")
    for q in range(B):
        ed, es, ec = merge_sorted([rows[q] for rows in per_index_q], limit, offset, descending)
        assert got[q].doc_ids.tolist() == ed.tolist(), (q, got[q].doc_ids, ed)
        assert got[q].scores.view(np.uint32).tolist() == es.view(np.uint32).tolist()
        assert got[q].count == ec


def test_merge_sorted_results_reference_pin():
    # src/tests/multi_index.rs:406-505: index 1 holds doc1 (priority 1), doc2 (3); index 2 doc3 (2), doc4 (4)
    def lists(order):
        desc = order == "DESC"
        a = sort_by_field([1, 2], [1.0, 1.0], [1, 2], [1.0, 3.0], 4, desc)
        b = sort_by_field([3, 4], [1.0, 1.0], [3, 4], [2.0, 4.0], 4, desc)
        key = {1: 1.0, 2: 3.0, 3: 2.0, 4: 4.0}
        return [([SearchHits(d, s, 2)], [np.asarray([key[x] for x in d.tolist()])]) for d, s in (a, b)]
    asc = ob.merge_sorted_index_results(lists("ASC"), 10, 0, "ASC")[0]
    assert asc.doc_ids.tolist() == [1, 3, 2, 4] and asc.count == 4
    desc = ob.merge_sorted_index_results(lists("DESC"), 10, 0, "DESC")[0]
    assert desc.doc_ids.tolist() == [4, 2, 3, 1] and desc.count == 4


def test_merge_sorted_results_equal_keys_go_to_the_lower_index():
    # MergeSortedIterator's strict comparison: on equal keys the first iterator's whole group comes first
    per = [([SearchHits(np.asarray([8, 9], np.uint64), np.asarray([1, 2], np.float32), 2)], [np.asarray([1.0, 1.0])]),
           ([SearchHits(np.asarray([2, 3], np.uint64), np.asarray([3, 4], np.float32), 2)], [np.asarray([1.0, 1.0])])]
    got = ob.merge_sorted_index_results(per, 3, 1)[0]
    assert got.doc_ids.tolist() == [9, 2, 3] and got.count == 4
    with pytest.raises(ValueError):
        ob.merge_sorted_index_results(per, 3, 0, "UP")
