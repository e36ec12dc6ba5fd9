"""sortBy cost on one GPU: oc_search_sorted next to oc_search on the same batches.

    python tools/bench_sort.py [--shape h1|t1|all] [--reps 20] [--out DIR]

Shapes (bench.py's synthetic corpora): h1 = hybrid, 1M docs x 768-d, vocab 200K, B = 256; t1 = fulltext, 10M docs,
vocab 1M, B = 256.  A `price` number field covers ~90 % of the documents (rounded gamma values: many ties).  Batches:
Zipf queries (bench.py's generator), a dense batch (every query = the corpus' most frequent term) and, on h1, a
match-all batch (term "": every term of the vocabulary, B = 4).  Per batch: device ms (CUDA events, oc_last_timing,
median of --reps calls after warm-up) of oc_search and of oc_search_sorted with the form chosen per query, forced walk
and forced gather (OC_SORT_FORM); which form each query took; and, from one torch.profiler pass, the share of the
sorted call's kernel time spent in the selection kernel (sort_select_kernel), with the call's kernels by time.  One
JSON line per shape."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import re  # noqa: E402

import oramacore_b200 as ob  # noqa: E402
from oramacore_b200 import synth  # noqa: E402
from oramacore_b200.types import MODE_FULLTEXT, MODE_HYBRID, TextQuery  # noqa: E402

with open(os.path.join(ROOT, "oramacore_b200", "csrc", "sort.cuh")) as _f:
    SORT_WALK_COST = float(re.search(r"SORT_WALK_COST = ([0-9.]+)f", _f.read()).group(1))

SHAPES = {
    "h1": dict(mode=MODE_HYBRID, n_docs=1_000_000, dim=768, vocab=200_000, batch=256),
    "t1": dict(mode=MODE_FULLTEXT, n_docs=10_000_000, dim=0, vocab=1_000_000, batch=256),
}


def _median_ms(ctx, fn, reps):
    for _ in range(3):
        fn()
    ms = []
    for _ in range(reps):
        fn()
        ms.append(ctx.last_timing()["device_ms"])
    return float(np.median(ms))


def _select_share(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    tot = sel = 0.0
    kernels = []
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        t = e.cuda_time_total if t is None else t
        if e.key.startswith(("Memcpy", "Memset", "cudaM")) or not t:
            continue
        tot += t
        kernels.append((e.key[:60], round(t / 1e3, 4)))
        if "sort_select_kernel" in e.key:
            sel += t
    kernels.sort(key=lambda x: -x[1])
    return sel / tot if tot else 0.0, sel / 1e3, kernels[:12]


def run_shape(name, reps, ctx):
    w = SHAPES[name]
    t0 = time.perf_counter()
    n = w["n_docs"]
    data = synth.make_text_corpus(n, w["vocab"])
    strs = ob.StringFieldStorage(ctx, data)
    emb = None
    if w["dim"]:
        emb = ob.EmbeddingFieldStorage(ctx, "BGEBase")
        emb.reserve(n)
        CH = 1 << 18
        for c0 in range(0, n, CH):
            c1 = min(n, c0 + CH)
            emb.insert_batch(np.arange(c0, c1, dtype=np.uint64), synth.make_vectors(c1 - c0, w["dim"], seed=synth.SEED_VECTORS + c0))
    rng = np.random.default_rng(5)
    has = rng.random(n) < 0.9
    price = np.round(rng.gamma(2.0, 30.0, size=n), 1)
    st = ob.SortStore(ctx, n)
    st.add_number_field("price", np.flatnonzero(has).astype(np.uint64), price[has])
    tsc = ob.TokenScoreContext(ctx, emb, strs)
    df = np.diff(data.fields[0].term_offsets.astype(np.int64))
    top = int(np.argmax(df))
    B = w["batch"]
    batches = {"zipf": synth.make_text_queries(w["vocab"], B), "dense": [TextQuery.single_terms([top])] * B}
    if name == "h1":
        batches["match_all"] = [TextQuery.from_tokens([[(0, t, 1.0) for t in range(w["vocab"])]])] * 4
    setup_s = time.perf_counter() - t0
    out = {"shape": name, "n_docs": n, "batch": B, "price_coverage": float(has.mean()), "setup_s": round(setup_s, 1),
           "switch": {"rule": "walk iff walk_cost * est_walk_entries <= bitmap_words + count", "walk_cost": SORT_WALK_COST},
           "batches": {}}
    for bname, texts in batches.items():
        b = len(texts)
        qv = None
        if emb is not None:
            qv = synth.make_vector_queries(synth.make_vectors(1 << 14, w["dim"]), b, seed=synth.SEED_VQUERIES)[0]
        kw = dict(texts=ob.TextQueryBatch(texts), q_vecs=qv)
        p = ob.TokenScoreParams(mode=w["mode"], limit_hint=10, similarity=0.0)
        res = {"queries": b, "df_top_term": int(df[top]) if bname == "dense" else None}
        res["search_device_ms"] = _median_ms(ctx, lambda: tsc.execute_batch(p, **kw), reps)
        counts = [h.count for h in tsc.execute_batch(p, **kw)]
        res["count_median"] = float(np.median(counts))
        sorted_call = lambda: ob.search_sorted(tsc, st, p, {"property": "price"}, **kw)  # noqa: E731
        for form in ("auto", "walk", "gather"):
            if form == "auto":
                os.environ.pop("OC_SORT_FORM", None)
            else:
                os.environ["OC_SORT_FORM"] = form
            res[f"sorted_device_ms_{form}"] = _median_ms(ctx, sorted_call, reps)
            if form == "auto":
                forms = ob.engine.sort_last_forms(ctx, b)
                res["forms_auto"] = {"walk": int((forms == 0).sum()), "gather": int((forms == 1).sum())}
                share, sel_ms, kernels = _select_share(sorted_call)
                res["select_kernel_share_of_kernel_time"] = round(share, 4)
                res["select_kernel_ms"] = round(sel_ms, 4)
                res["kernel_ms_profiled"] = kernels
        os.environ.pop("OC_SORT_FORM", None)
        res["sorted_over_search"] = round(res["sorted_device_ms_auto"] / res["search_device_ms"], 3)
        out["batches"][bname] = res
        print(json.dumps({"shape": name, "batch": bname, **res}), flush=True)
    st.close(); strs.close()
    if emb is not None:
        emb.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="all", choices=["all"] + sorted(SHAPES))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None, help="directory for r03_sort_<shape>.json")
    args = ap.parse_args()
    ctx = ob.Context(0)
    info = ctx.device_info()
    try:
        import subprocess
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    except OSError:
        q = ""
    for name in (sorted(SHAPES) if args.shape == "all" else [args.shape]):
        line = {"tool": "bench_sort", "device": info["name"], "nvidia_smi": q, **run_shape(name, args.reps, ctx)}
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"r03_sort_{name}.json"), "w") as f:
                f.write(json.dumps(line) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
