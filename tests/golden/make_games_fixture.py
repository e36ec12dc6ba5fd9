"""Generates tests/golden/games_fulltext.npz — BASELINE configs[0], "benches/fulltext_simple.rs on
games.json": the reference's own CPU-runnable plumbing case.

    python tests/golden/make_games_fixture.py <oramacore checkout>/benches/games.json

The tests read only the fixture, never games.json.  The fixture holds only DERIVED integer / float
arrays — the committed postings of the 1512 game documents (fields title, description) as laid out
by oramacore_b200.hostindex (lower-case alphanumeric tokenizer; the reference's stemmer lives in an un-vendored crate), the resolved term lists of a query
set (the bench's own strings + game-domain ones, prefix and exact resolution), and the ORACLE's answers
(count, top-10 doc ids and scores).  tests/test_gpu_zz_games_config0.py checks the oracle against the stored
answers on the CPU and the GPU path against the oracle on a B200."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import oracle as orc                                   # noqa: E402
from oramacore_b200.hostindex import HostStringIndex   # noqa: E402

QUERIES = [  # (term, exact, on the GPU test too?)  benches/fulltext_simple.rs:438-458 use the first three strings
    ("technology", False, False), ("technology software", False, False), ("development", False, False),
    ("fantasy", False, True), ("open world", False, True), ("rpg", True, True), ("adventure", False, True),
    ("elden ring", True, True), ("war", False, True), ("space station", False, True), ("racing cars", False, False),
    ("zzzunknownterm", False, False), ("the", False, False),
]


def main():
    games = json.load(open(sys.argv[1]))
    h = HostStringIndex(("title", "description"))
    for i, g in enumerate(games):
        h.insert(i, {"title": g.get("title", ""), "description": g.get("description", "")})
    data = h.commit()
    out = {"n_rows": np.int64(data.n_rows), "document_count": np.int64(data.document_count), "n_fields": np.int64(len(data.fields))}
    for fi, f in enumerate(data.fields):
        out[f"f{fi}_avg"] = np.float32(f.avg_field_len)
        out[f"f{fi}_offs"] = f.term_offsets.astype(np.uint64)
        out[f"f{fi}_row"] = f.post_row.astype(np.uint32)
        out[f"f{fi}_tf"] = f.post_tf.astype(np.uint16)
        out[f"f{fi}_len"] = f.post_len.astype(np.uint16)
    ix = orc.StrIndex(data)
    sb = orc.SearchBatch(ix, None)
    qs = []
    for term, exact, _ in QUERIES:
        q = h.resolve(term, exact=exact)
        qs.append(q)
        sb.add(0, limit=10, text=q)
    od, os_, on, oc = sb.run(4)
    out["n_queries"] = np.int64(len(qs))
    out["gpu_ok"] = np.asarray([g for _, _, g in QUERIES], np.uint8)
    out["exact"] = np.asarray([e for _, e, _ in QUERIES], np.uint8)
    for i, q in enumerate(qs):
        out[f"q{i}_tto"] = q.token_term_offsets
        out[f"q{i}_field"] = q.term_field
        out[f"q{i}_term"] = q.term_id
        out[f"q{i}_w"] = q.term_weight
        print(f"{QUERIES[i][0]!r:24} exact={QUERIES[i][1]!s:5} tokens={q.n_tokens} terms={len(q.term_id):4d} count={int(oc[i]):4d} "
              f"top={od[i, :min(3, on[i])].tolist()}")
    out["exp_docs"], out["exp_scores"], out["exp_n"], out["exp_count"] = od, os_, on, oc
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "games_fulltext.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes;", sum(int(f.term_offsets[-1]) for f in data.fields), "postings")


if __name__ == "__main__":
    main()
