"""BASELINE configs[0] — "benches/fulltext_simple.rs on games.json (CPU-only reference, plumbing)":
fulltext search over the 1512 game documents (fields title + description) for the bench's own query
strings and a few game-domain ones.  The corpus travels as a derived fixture (committed postings +
resolved query terms + the oracle's answers; tests/golden/make_games_fixture.py), so the test needs
nothing outside the repository."""
import os

import numpy as np
import pytest

import oramacore_b200 as ob
from helpers import assert_topk_equal

FIX = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "games_fulltext.npz")


def _load():
    z = np.load(FIX)
    fields = [ob.FieldPostings(float(z[f"f{i}_avg"]), z[f"f{i}_offs"], z[f"f{i}_row"], z[f"f{i}_tf"], z[f"f{i}_len"])
              for i in range(int(z["n_fields"]))]
    data = ob.StringIndexData(fields, int(z["n_rows"]), int(z["document_count"]), None)
    qs = [ob.TextQuery(z[f"q{i}_tto"], z[f"q{i}_field"], z[f"q{i}_term"], z[f"q{i}_w"]) for i in range(int(z["n_queries"]))]
    return z, data, qs


def test_oracle_reproduces_the_committed_answers(orc):
    z, data, qs = _load()
    assert data.n_rows == 1512 and sum(int(f.term_offsets[-1]) for f in data.fields) == 95107
    sb = orc.SearchBatch(orc.StrIndex(data), None)
    for q in qs:
        sb.add(0, limit=10, text=q)
    od, os_, on, oc = sb.run(2)
    assert np.array_equal(oc, z["exp_count"]) and np.array_equal(on, z["exp_n"])
    for i in range(len(qs)):
        assert np.array_equal(od[i, :on[i]], z["exp_docs"][i, :on[i]])
        assert np.array_equal(os_[i, :on[i]], z["exp_scores"][i, :on[i]])       # same C code, same bits
    # shape of the plumbing case: "technology" matches 20 games, "the" almost all, an unknown term none
    assert int(oc[0]) == 20 and int(oc[-1]) == 1468 and int(oc[-2]) == 0


# Written after this round's GPU budget was spent: it only uses API paths the other GPU parity tests
# exercise (multi-field, multi-term tokens, df counted on device) and is expected to pass, but until it has
# run once on a B200 it must not be able to turn the GPU tier red (the file also sorts last).  Remove the
# marker when it shows up as XPASS.

@pytest.mark.gpu
def test_gpu_fulltext_on_the_games_corpus(gpu_ctx, orc):
    z, data, qs = _load()
    sel = [i for i in range(len(qs)) if z["gpu_ok"][i]]
    strs = ob.StringFieldStorage(gpu_ctx, data)
    hits = ob.search(gpu_ctx, None, strs, "fulltext", texts=[qs[i] for i in sel], limit=10)
    for h, i in zip(hits, sel):
        n = int(z["exp_n"][i])
        assert h.count == int(z["exp_count"][i]), (i, h.count, int(z["exp_count"][i]))
        assert_topk_equal(h.doc_ids, h.scores, z["exp_docs"][i, :n], z["exp_scores"][i, :n], atol=1e-5)
    strs.close()
