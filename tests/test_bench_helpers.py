"""bench.py's fp64 recall checkers against the C oracle on small corpora (CPU)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from oramacore_b200 import synth


def test_fp64_vector_topk_matches_oracle_f64(orc):
    rows = synth.make_clustered_vectors(3000, 96, n_centroids=20, seed=3)
    qv, _ = synth.make_vector_queries(rows, 9, seed=4)
    vi, vs = bench.fp64_vector_topk(rows, qv, 10, chunk=700)
    st = orc.EmbStore(rows)
    for i in range(9):
        ed, ec = orc.vector_f64(st, qv[i], 10)
        assert np.allclose(vs[i], ec, atol=1e-12)
        assert set(vi[i].tolist()) == set(int(x) for x in ed)


def test_fp64_hybrid_topk_close_to_fp32_oracle(orc):
    n, dim, vocab = 4000, 64, 300
    rows = synth.make_vectors(n, dim, seed=5)
    qv, _ = synth.make_vector_queries(rows, 12, seed=6)
    data = synth.make_text_corpus(n, vocab, seed=7)
    texts = synth.make_text_queries(vocab, 12, seed=8)
    vi, vs = bench.fp64_vector_topk(rows, qv, 10)
    ix, st = orc.StrIndex(data), orc.EmbStore(rows)
    sb = orc.SearchBatch(ix, st)
    for i in range(12):
        sb.add(2, limit=10, similarity=-1.0, q_vec=qv[i], text=texts[i])
    od, os_, on, oc = sb.run(2)
    for i in range(12):
        ed, es = bench.fp64_hybrid_topk(data, texts[i], vi[i], vs[i], 10)
        assert np.allclose(es, os_[i, :on[i]], atol=2e-5), (es, os_[i])
        hit, tot = bench.recall_hits(od[i, :on[i]], ed, es, os_[i, :on[i]])
        assert hit == tot


def test_dump_outputs_writes_the_step_arrays(tmp_path, monkeypatch):
    rng = np.random.default_rng(9)
    B, limit = 40, 10
    raw = (rng.integers(0, 1 << 40, (B, limit), dtype=np.uint64), rng.random((B, limit), dtype=np.float32),
           rng.integers(0, limit + 1, B).astype(np.uint32), rng.integers(0, 1 << 30, B).astype(np.uint64))
    bench.dump_outputs(str(tmp_path / "all"), raw)
    got = {n: np.load(tmp_path / "all" / f"{n}.npy") for n in ("doc_ids", "scores", "n", "count")}
    assert sorted(os.listdir(tmp_path / "all")) == ["count.npy", "doc_ids.npy", "n.npy", "scores.npy"]
    assert got["scores"].dtype == np.float32 and np.array_equal(got["scores"], raw[1])
    for name, a in zip(("doc_ids", "n", "count"), (raw[0], raw[2], raw[3])):
        assert got[name].dtype == np.float64 and np.array_equal(got[name].astype(np.uint64), a)

    # over the size cap: the same seeded sample of queries every time, named by query_index
    cap = 10 * (limit * 12 + 24) + 5 * 128
    monkeypatch.setattr(bench, "DUMP_CAP_BYTES", cap)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), raw)
    idx = np.load(tmp_path / "s1" / "query_index.npy")
    assert idx.shape == (10,) and np.array_equal(idx, np.load(tmp_path / "s2" / "query_index.npy"))
    rows = idx.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "s1" / "doc_ids.npy").astype(np.uint64), raw[0][rows])
    assert np.array_equal(np.load(tmp_path / "s1" / "scores.npy"), raw[1][rows])
    assert sum(os.path.getsize(tmp_path / "s1" / f) for f in os.listdir(tmp_path / "s1")) <= cap
