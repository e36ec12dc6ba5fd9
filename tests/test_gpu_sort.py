"""sortBy on the GPU (oc_search_sorted) against (1) the reference's pinned answers (src/tests/sort.rs: number :8-110,
date :113-218, bool :220-323, unknown field :325-353, filter with one shared key :418-493; src/tests/multi_index.rs:406-505
through merge_sorted_index_results) and (2) the numpy statement of sort_token_scores_by_field + truncate (sort_spec.py)
over the oracle's score maps, in fulltext, vector and hybrid mode, with both selection forms (OC_SORT_FORM).  Scores:
bit-identical to the oracle's map values in fulltext mode; with vector scores, within the parity tests' tolerance of
the oracle and bit-identical to what oc_search returns for the same documents."""
import os

import numpy as np
import pytest

import oramacore_b200 as ob
from helpers import build_index
from oramacore_b200 import filters as F
from oramacore_b200 import synth
from oramacore_b200.types import MODE_FULLTEXT, MODE_HYBRID, MODE_VECTOR, TextQuery
from sort_spec import sort_by_field

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["walk", "gather"])
def form(request):
    old = os.environ.get("OC_SORT_FORM")
    os.environ["OC_SORT_FORM"] = request.param
    yield request.param
    if old is None:
        os.environ.pop("OC_SORT_FORM")
    else:
        os.environ["OC_SORT_FORM"] = old


def _ft(ctx, h):
    return ob.TokenScoreContext(ctx, None, ob.StringFieldStorage(ctx, h.data))


def _ids(hits):
    return hits.doc_ids.tolist()


def test_reference_pins_number_date_bool(gpu_ctx, form):
    # sort.rs:8-323: documents 1 and 2, term "" (every document), order defaults to ASC
    h = build_index([(1, {"text": "Tommaso"}), (2, {"text": "Michele"})])
    tsc = _ft(gpu_ctx, h)
    st = ob.SortStore(gpu_ctx, 3)
    st.add_number_field("year", [1, 2], [1990, 1994])
    st.add_date_field("birthday", [1, 2], [631152000000, 757382400000])   # 1990-01-01, 1994-01-01 (ms)
    st.add_bool_field("is_good", [2], [1])
    p = ob.TokenScoreParams(mode=MODE_FULLTEXT)
    for prop in ("year", "birthday", "is_good"):
        for sort_by, exp in (({"property": prop}, [1, 2]), ({"property": prop, "order": "ASC"}, [1, 2]),
                             ({"property": prop, "order": "DESC"}, [2, 1])):
            r = ob.search_sorted(tsc, st, p, sort_by, texts=[h.resolve("")])[0]
            assert _ids(r) == exp and r.count == 2, (prop, sort_by, _ids(r))
    hits, keys = ob.search_sorted(tsc, st, p, {"property": "is_good", "order": "DESC"}, texts=[h.resolve("")], with_keys=True)
    assert keys[0].tolist() == [1.0, 0.0]
    # sort.rs:325-353: an unknown property is SortFieldNotFound; at the ABI an unknown field id is OC_ERR_INVALID
    with pytest.raises(KeyError):
        ob.search_sorted(tsc, st, p, {"property": "unknown_field"}, texts=[h.resolve("")])
    st.fields["ghost"] = 99
    with pytest.raises(ob.OcError) as e:
        ob.search_sorted(tsc, st, p, {"property": "ghost"}, texts=[h.resolve("")])
    assert e.value.code == -1
    st.close(); tsc.str.close()


def test_reference_pin_filter_with_one_shared_key(gpu_ctx, form):
    # sort.rs:418-493: number = 2 everywhere, where is_active = true keeps 1 and 3
    h = build_index([(1, {"text": "Document One"}), (2, {"text": "Document Two"}), (3, {"text": "Document Three"})])
    tsc = _ft(gpu_ctx, h)
    st = ob.SortStore(gpu_ctx, 4)
    st.add_number_field("number", [1, 2, 3], [2.0, 2.0, 2.0])
    p = ob.TokenScoreParams(mode=MODE_FULLTEXT, filtered_doc_ids=F.to_bitmap(F.Ids([1, 3]), 4), filter_nbits=4)
    r = ob.search_sorted(tsc, st, p, {"property": "number", "order": "ASC"}, texts=[h.resolve("")])[0]
    assert r.count == 2 and _ids(r) == [1, 3]
    st.close(); tsc.str.close()


def test_reference_pin_multi_index(gpu_ctx, form):
    # multi_index.rs:406-505: index 1 = doc1 (priority 1), doc2 (3); index 2 = doc3 (2), doc4 (4)
    parts = [[(1, 1.0), (2, 3.0)], [(3, 2.0), (4, 4.0)]]
    for order, exp in (("ASC", [1, 3, 2, 4]), ("DESC", [4, 2, 3, 1])):
        per = []
        for docs in parts:
            h = build_index([(d, {"text": "item"}) for d, _ in docs])
            tsc = _ft(gpu_ctx, h)
            st = ob.SortStore(gpu_ctx, 5)
            st.add_number_field("priority", [d for d, _ in docs], [v for _, v in docs])
            p = ob.TokenScoreParams(mode=MODE_FULLTEXT, limit_hint=10, vector_limit=10)
            per.append(ob.search_sorted(tsc, st, p, {"property": "priority", "order": order}, texts=[h.resolve("item")], with_keys=True))
            st.close(); tsc.str.close()
        r = ob.merge_sorted_index_results(per, 10, 0, order)[0]
        assert _ids(r) == exp and r.count == 4


def _same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    nan = np.isnan(a)
    return a.shape == b.shape and bool(np.all(nan == np.isnan(b))) and a[~nan].view(np.uint32).tolist() == b[~nan].view(np.uint32).tolist()


@pytest.mark.parametrize("mode,sparse_ids", [(MODE_FULLTEXT, False), (MODE_FULLTEXT, True), (MODE_VECTOR, False),
                                              (MODE_HYBRID, False), (MODE_HYBRID, True)])
def test_random_corpus_against_the_oracle_score_maps(gpu_ctx, orc, form, mode, sparse_ids):
    n, dim, vocab, B = 40000, 384, 3000, 10
    rng = np.random.default_rng(17)
    rows = synth.make_vectors(n, dim, seed=71)
    qv, _ = synth.make_vector_queries(rows, B, seed=72)
    data = synth.make_text_corpus(n, vocab, seed=73)
    texts = synth.make_text_queries(vocab, B - 2, seed=74)
    texts.append(TextQuery.from_tokens([[(0, t, 1.0) for t in range(vocab)]]))                  # "": every term
    texts.append(TextQuery.from_tokens([[(0, t, 1.0) for t in range(40, 60)], [(0, 7, 1.0)]]))    # a prefix + a term
    ids = (np.arange(n, dtype=np.uint64) * 3 + 2) if sparse_ids else np.arange(n, dtype=np.uint64)
    if sparse_ids:
        data.row_doc_ids = ids
    nbits = int(ids.max()) + 1
    emb = ob.EmbeddingFieldStorage(gpu_ctx, "BGESmall")
    emb.insert_batch(ids, rows)
    strs = ob.StringFieldStorage(gpu_ctx, data)
    gone = [5, 77, 4000]
    strs.delete(ids[gone]); emb.delete(ids[gone])                 # uncommitted deletes stay out of the map
    deleted = np.zeros(n, np.uint8); deleted[gone] = 1
    tsc = ob.TokenScoreContext(gpu_ctx, emb if mode != MODE_FULLTEXT else None, strs if mode != MODE_VECTOR else None)
    has = rng.random(n) < 0.9                                     # documents without a price are never emitted
    price = np.round(rng.gamma(2.0, 10.0, size=n))                # heavy ties
    stamp = rng.integers(-2**40, 2**40, size=n)
    st = ob.SortStore(gpu_ctx, nbits)
    st.add_number_field("price", ids[has], price[has])
    st.add_date_field("created", ids[has], stamp[has])
    ix = orc.StrIndex(data)
    est = orc.EmbStore(rows, row_doc_ids=ids, deleted=deleted)
    where_ids = ids[rng.random(n) < 0.6]
    omc_doc = np.sort(rng.choice(ids, 500, replace=False)).astype(np.uint64)
    omc_mult = rng.uniform(0.5, 2.0, 500).astype(np.float32)
    variants = [dict(limit=10, offset=0), dict(limit=1000, offset=24, where=True), dict(limit=20, offset=5, threshold=0.5),
                dict(limit=30, offset=3, omc=True)]
    if mode == MODE_HYBRID:   # a negative score makes the hybrid minimum negative: OMC then re-runs the tile scorer
        neg = [TextQuery(t.token_term_offsets, t.term_field, t.term_id, np.where(np.arange(t.term_id.shape[0]) == 0, -1.0, 1.0).astype(np.float32))
               for t in texts]
        variants.append(dict(limit=15, offset=0, omc=True, texts=neg))
    alive_ids = ids[deleted == 0]
    for vi, v in enumerate(variants):
        qt = v.get("texts", texts)
        where = v.get("where", False)
        p = ob.TokenScoreParams(mode=mode, limit_hint=v["limit"], offset=v["offset"], similarity=0.0, threshold=v.get("threshold"),
                                filtered_doc_ids=orc.make_filter_bits(where_ids.tolist(), nbits) if where else None,
                                filter_nbits=nbits if where else 0,
                                omc_doc_ids=omc_doc if v.get("omc") else None, omc_mult=omc_mult if v.get("omc") else None)
        kw = dict(texts=qt if mode != MODE_VECTOR else None, q_vecs=qv if mode != MODE_FULLTEXT else None)
        plain = tsc.execute_batch(p, **kw)
        for prop, vals, desc in (("price", price, False), ("price", price, True), ("created", stamp, vi % 2 == 0)):
            got = ob.search_sorted(tsc, st, p, {"property": prop, "order": "DESC" if desc else "ASC"}, **kw)
            forms = ob.engine.sort_last_forms(gpu_ctx, B)
            assert forms.tolist() == [0 if form == "walk" else 1] * B
            vlimit = v["limit"]
            ft_allowed = np.intersect1d(alive_ids, where_ids) if where else alive_ids
            for q in range(B):
                if mode == MODE_VECTOR:
                    m = orc.vector(est, qv[q], vlimit, 0.0, *((orc.make_filter_bits(where_ids.tolist(), nbits), nbits) if where else ()))
                else:
                    m = orc.fulltext(ix, qt[q], threshold=v.get("threshold"), filter_bits=orc.make_filter_bits(ft_allowed.tolist(), nbits),
                                     filter_nbits=nbits)
                    if mode == MODE_HYBRID:
                        vm = orc.vector(est, qv[q], vlimit, 0.0, *((orc.make_filter_bits(where_ids.tolist(), nbits), nbits) if where else ()))
                        m = orc.hybrid_combine(vm, m)
                if v.get("omc"):
                    m = orc.apply_omc(m, omc_doc, omc_mult)
                ed, es = sort_by_field(m[0], m[1], ids[has], vals[has], v["limit"] + v["offset"], desc)
                ed, es = ed[v["offset"]:], es[v["offset"]:]
                tag = (vi, prop, desc, q)
                assert got[q].count == plain[q].count == m[0].shape[0], tag
                assert _ids(got[q]) == ed.tolist(), (tag, got[q].doc_ids[:8], ed[:8])
                if mode == MODE_FULLTEXT:   # BM25 scores are bit-identical to the oracle's
                    assert _same_bits(got[q].scores, es), (tag, got[q].scores[:8], es[:8])
                else:   # cosine scores carry the vector stage's rounding (the parity tests' tolerance) ...
                    assert np.allclose(got[q].scores, es, rtol=0, atol=1e-5, equal_nan=True), (tag, got[q].scores[:8], es[:8])
                # ... and every hit oc_search also returns carries the very same value
                common = {d: s for d, s in zip(_ids(plain[q]), plain[q].scores.tolist())}
                both = [(common[d], s) for d, s in zip(_ids(got[q]), got[q].scores.tolist()) if d in common]
                assert _same_bits([a for a, _ in both], [b for _, b in both]), (tag, both[:4])
    st.close(); emb.close(); strs.close()


def test_default_form_choice_and_errors(gpu_ctx):
    # without OC_SORT_FORM each query picks its form from its count: a match-all query walks, a rare term gathers
    assert "OC_SORT_FORM" not in os.environ
    n, vocab = 200000, 20000
    data = synth.make_text_corpus(n, vocab, seed=81)
    strs = ob.StringFieldStorage(gpu_ctx, data)
    tsc = ob.TokenScoreContext(gpu_ctx, None, strs)
    st = ob.SortStore(gpu_ctx, n)
    rng = np.random.default_rng(3)
    st.add_number_field("price", np.arange(n, dtype=np.uint64), rng.random(n))
    texts = [TextQuery.from_tokens([[(0, t, 1.0) for t in range(vocab)]]), TextQuery.single_terms([vocab - 1])]
    r = ob.search_sorted(tsc, st, ob.TokenScoreParams(mode=MODE_FULLTEXT), {"property": "price"}, texts=texts)
    assert ob.engine.sort_last_forms(gpu_ctx, 2).tolist() == [0, 1], r
    with pytest.raises(ob.OcError) as e:   # a document listed twice in one field
        st.add_number_field("dup", [1, 1], [1.0, 2.0])
    assert e.value.code == -1
    with pytest.raises(ob.OcError):
        st.add_number_field("nan", [1], [float("nan")])
    with pytest.raises(ob.OcError) as e:
        ob.search_sorted(tsc, st, ob.TokenScoreParams(mode=MODE_FULLTEXT, sharded=True), {"property": "price"}, texts=texts)
    assert e.value.code == -4
    st.close(); strs.close()
