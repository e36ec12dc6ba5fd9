#!/usr/bin/env python
"""bench.py — the hot path of BASELINE.json's metric on synthetic corpora of the named shape.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload h1|h1c|v1|t1|v2] [--batch B]
    python bench.py --impl reference ...      # the CPU restatement (oracle) on the host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's results (see dump_outputs)

A "step" = one pass of the hot path over one batch of B queries through the C ABI
(oc_search): hybrid = embedding scan + BM25 posting scorer + fusion/top-k.  N_BATCHES distinct
query batches rotate through the timed loop (no step replays the previous step's inputs).
  value : whole-job QPS with inputs resident in HBM — B*K / sum of the library's own
          CUDA-event device time (H2D of queries .. last kernel), max over ranks.
  e2e   : QPS through the public call with HOST buffers (H2D + kernels + D2H inside),
          K calls bracketed by barrier + device synchronize, max over ranks.
Under torchrun (N>1) the corpus is sharded by document across ranks (strong scaling: the
named corpus is fixed); one NCCL all-gather of per-shard top-k per batch, merged on device.
The matrix (3.07 GB at 1M x 768) is far larger than L2 (126 MB), so no L2 flush is needed
between iterations.
After the timed region (never inside it): parity of the timed queries against the CPU oracle
(at every N: rank 0 runs the oracle on the UNSHARDED corpus and every rank's answer must be
byte-identical to rank 0's), recall@10 against an fp64 evaluation on >= 1000 queries, the CPU
baseline, and — single GPU, h1 — a driver-visible sub-result for BASELINE configs[1] (B = 1 scan)
under "extra".
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_BATCHES = 8   # distinct query batches rotated through the timed loop

WORKLOADS = {
    # BASELINE.json configs[3] (the config the hybrid-QPS metric is quoted on), configs[1], configs[2], configs[4]
    "h1": dict(mode="hybrid", n_docs=1_000_000, dim=768, vocab=200_000, batch=256,
               desc="hybrid vector+BM25, 1M docs x 768-d fp32, cosine+BM25F top-10 (BASELINE configs[3])"),
    "h1c": dict(mode="hybrid", n_docs=1_000_000, dim=768, vocab=200_000, batch=256, clustered=True,
                desc="hybrid vector+BM25, 1M docs x 768-d fp32 in 2000 near-duplicate clusters (within-cluster cosine 0.99), "
                     "cosine+BM25F top-10 (configs[3] shape, adversarial embedding distribution)"),
    "v1": dict(mode="vector", n_docs=1_000_000, dim=768, vocab=0, batch=1,
               desc="1M x 768-d fp32 embeddings, cosine top-10, batch=1 (BASELINE configs[1])"),
    "t1": dict(mode="fulltext", n_docs=10_000_000, dim=0, vocab=1_000_000, batch=256,
               desc="BM25 fulltext, 10M synthetic docs (Zipf), batch=256 (BASELINE configs[2])"),
    "v2": dict(mode="vector", n_docs=10_000_000, dim=1024, vocab=0, batch=1024, dtype="bf16",
               desc="10M x 1024-d bf16 embeddings, cosine top-10, batch=1024 (BASELINE configs[4])"),
}

# oc_timing.scan_variant (include/oramacore_b200.h OC_SCAN_*) -> (kernel, description)
SCAN_VARIANTS = {
    0: ("emb_scan_kernel", "exact fp32 sweep"),
    1: ("emb_gemm_kernel", "tcgen05 kind::tf32 on the fp32 rows + exact fp32 re-score"),
    2: ("emb_gemm_pair_kernel", "tcgen05 cta_group::2 kind::tf32 on the fp32 rows + exact fp32 re-score"),
    3: ("emb_gemm_cvt_kernel", "tcgen05 cta_group::2 kind::f16, fp32 rows streamed once and rounded to bf16 in the SM, + exact fp32 re-score"),
    4: ("emb_gemm_kernel", "tcgen05 kind::f16 on the bf16 rows + exact fp32 re-score"),
    5: ("emb_gemm_pair_kernel", "tcgen05 cta_group::2 kind::f16 on the bf16 rows + exact fp32 re-score"),
}
METRIC = {"h1": "hybrid_search_qps_at_recall10_ge_0.99_1Mx768", "h1c": "hybrid_search_qps_clustered_1Mx768"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="h1", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--n-docs", type=int, default=0, help="override corpus size (debug)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU baseline / parity sample budget")
    ap.add_argument("--recall-queries", type=int, default=1024, help="queries of the fp64 recall check")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip oracle parity, recall and the CPU baseline")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[1] sub-result of the h1 line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's results as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200 (the reference leg times a load-dependent sample)")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_workload(w, n_docs, batch, rank, world, keep_all):
    """Synthetic corpus of the named shape; shard = contiguous doc-row range (SURVEY.md §8e).
    N_BATCHES query batches: batch i is drawn with seed + i.  keep_all: keep the unsharded
    matrix on this rank (rank 0: parity and recall are checked against the whole corpus)."""
    from oramacore_b200 import synth
    lo, hi = (n_docs * rank) // world, (n_docs * (rank + 1)) // world
    out = dict(lo=lo, hi=hi)
    if w["dim"] and w.get("dtype") == "bf16":
        # too large to hold in fp32 on the host: rows are generated chunk by chunk at load time (see main);
        # queries are planted on rows of the first chunk
        first = synth.make_vectors(min(n_docs, 1 << 18), w["dim"])
        qb = [synth.make_vector_queries(first, batch, seed=synth.SEED_VQUERIES + i) for i in range(N_BATCHES)]
        out.update(rows=None, qv=[q for q, _ in qb], planted=[j for _, j in qb], chunked=True)
    elif w["dim"]:
        gen = synth.make_clustered_vectors if w.get("clustered") else synth.make_vectors
        rows = gen(n_docs, w["dim"])          # deterministic: every rank draws the same stream
        qb = [synth.make_vector_queries(rows, batch, seed=synth.SEED_VQUERIES + i) for i in range(N_BATCHES)]
        # rows = this rank's shard (a view when the whole matrix stays resident on this rank)
        out.update(rows=rows[lo:hi] if (keep_all or world == 1) else rows[lo:hi].copy(),
                   rows_all=rows if (keep_all or world == 1) else None,
                   qv=[q for q, _ in qb], planted=[j for _, j in qb])
        del rows
    if w["vocab"]:
        data = synth.make_text_corpus(n_docs, w["vocab"])
        out.update(data_all=data, texts=[synth.make_text_queries(w["vocab"], batch, seed=synth.SEED_TQUERIES + i)
                                         for i in range(N_BATCHES)])
    return out


def config_of(w, batch, n_docs, world=1):
    return {"workload": w["desc"], "batch": batch, "n_docs": n_docs, "dim": w["dim"], "vocab": w["vocab"],
            "limit": 10, "similarity": 0.0, "query_batches_rotated": N_BATCHES}


def run_reference(args, w, batch, n_docs):
    """--impl reference: the reference's CPU algorithm (oracle port; the Rust reference cannot be
    built here) on all host cores, each step a bounded sample of the same workload."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    wl = make_workload(w, n_docs, batch, 0, 1, True)
    cores = os.cpu_count() or 1
    ix = orc.StrIndex(wl["data_all"]) if w["vocab"] else None
    st = orc.EmbStore(wl["rows"]) if w["dim"] else None
    mode = {"fulltext": 0, "vector": 1, "hybrid": 2}[w["mode"]]
    sample = min(batch, max(cores, 8))
    threads = cores

    def one_step(k):
        sb = orc.SearchBatch(ix, st)
        nb = k % N_BATCHES
        for i in range(sample):
            j = ((k // N_BATCHES) * sample + i) % batch
            sb.add(mode, limit=10, similarity=0.0, q_vec=wl["qv"][nb][j] if w["dim"] else None,
                   text=wl["texts"][nb][j] if w["vocab"] else None)
        t0 = time.perf_counter()
        sb.run(threads)
        return time.perf_counter() - t0

    # bound the run to a few minutes: a step is one query per thread; when a full-width step is too
    # long for steps+warmup of them (the scan is DRAM-bound on the host, so time ~ queries in flight),
    # shrink the per-step sample and the thread count together and report the threads actually used
    t_probe = one_step(0)
    budget = 150.0
    n_steps_total = args.steps + max(args.warmup - 1, 0)
    if t_probe * n_steps_total > budget:
        scale = budget / (t_probe * n_steps_total)
        sample = threads = max(8, min(sample, int(sample * scale)))
    for k in range(1, args.warmup):
        one_step(k)
    times = [one_step(k) for k in range(args.steps)]
    total = sum(times)
    qps = sample * args.steps / total
    cores = threads
    cfg = config_of(w, batch, n_docs)
    cfg["sample_queries_per_step"] = sample
    line = {"impl": "reference",
            "metric": METRIC.get(args.workload, f"{w['mode']}_search_qps"),
            "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
                             "sample": f"{sample} queries/step x {args.steps} steps, one query per thread; C restatement "
                                       "of the reference algorithm (brute-force scan + hash-map BM25), not the Rust binary"},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# fp64 recall oracle (checker; numpy).  Vector: exact fp64 cosine top-k by blocked dgemm.  Hybrid:
# BM25F in fp64 over the same postings + the reference's fusion (token_score.rs:393-422) in fp64.
# ------------------------------------------------------------------------------------------------
def fp64_vector_topk(rows, qv, k, chunk=65536):
    """Exact fp64 cosine top-k of every query over all rows: blocked dgemm + per-row top-k (torch on the
    host: both are multi-threaded; this is a checker, nothing here touches the GPU)."""
    import torch
    Q = torch.from_numpy(np.ascontiguousarray(qv)).double()
    Q = Q / Q.norm(dim=1, keepdim=True).clamp_min(1e-300)
    nq = Q.shape[0]
    bs = torch.full((nq, k), -float("inf"), dtype=torch.float64)
    bi = torch.zeros((nq, k), dtype=torch.int64)
    for c0 in range(0, rows.shape[0], chunk):
        X = torch.from_numpy(rows[c0:c0 + chunk]).double()
        X = X / X.norm(dim=1, keepdim=True).clamp_min(1e-300)
        S = Q @ X.T
        s, i = S.topk(min(k, S.shape[1]), dim=1)
        cs, ci = torch.cat([bs, s], 1), torch.cat([bi, i + c0], 1)
        o = cs.argsort(dim=1, descending=True, stable=True)[:, :k]
        bs, bi = cs.gather(1, o), ci.gather(1, o)
    return bi.numpy(), bs.numpy()


def fp64_hybrid_topk(data, text, v_idx, v_cos, k, bm25_k=1.2, b=0.75, scratch=None):
    """One query: (doc ids, scores) of the fp64 hybrid top-k; single-term tokens, one field.
    BM25F in fp64 over the same postings + the reference's fusion (token_score.rs:393-422).
    scratch: a zeroed float64 array of n_rows reused across calls (left zeroed)."""
    f = data.fields[0]
    N = float(data.document_count)
    ft_dense = scratch if scratch is not None else np.zeros(int(data.n_rows))
    touched = []
    for t in text.term_id.tolist():
        lo, hi = int(f.term_offsets[t]), int(f.term_offsets[t + 1])
        if hi == lo:
            continue
        df = hi - lo
        idf = np.log1p((N - df + 0.5) / (df + 0.5))
        tf = f.post_tf[lo:hi].astype(np.float64)
        ln = f.post_len[lo:hi].astype(np.float64)
        S = tf / (1.0 - b + b * (ln / f.avg_field_len))
        r = f.post_row[lo:hi]
        ft_dense[r] += idf * (bm25_k + 1.0) * S / (bm25_k + S)     # rows are unique inside a term
        touched.append(r)
    if touched:
        u = np.concatenate(touched)
        ft = ft_dense[u]
    else:
        u, ft = np.zeros(0, np.int64), np.zeros(0)
    mx = max(0.0, ft.max() if ft.size else 0.0, v_cos.max() if v_cos.size else 0.0)
    mn = min(0.0, ft.min() if ft.size else 0.0, v_cos.min() if v_cos.size else 0.0)
    den = mx - mn
    kk = min(3 * k, ft.shape[0])           # a row may be listed once per term it holds: 3k covers k distinct rows
    cand = {}
    if kk:
        top = np.argpartition(-ft, kk - 1)[:kk]
        for i in top.tolist():
            cand[int(u[i])] = (float(ft[i]) - mn) / den
    for r, c in zip(v_idx.tolist(), v_cos.tolist()):
        fv = float(ft_dense[r])
        cand[int(r)] = ((fv - mn) / den if fv != 0.0 else 0.0) + (c - mn) / den
    if touched:
        ft_dense[u] = 0.0
    items = sorted(cand.items(), key=lambda kv: (-kv[1], kv[0]))[:k]
    return [d for d, _ in items], [s for _, s in items]


def recall_hits(got_docs, exp_docs, exp_scores, got_scores):
    """recall@k with boundary ties counted as hits (SURVEY §8d: |dscore| <= 1e-6 at the boundary)."""
    g = set(int(x) for x in got_docs)
    hit = 0
    for d, s in zip(exp_docs, exp_scores):
        hit += (int(d) in g) or abs(s - exp_scores[-1]) <= 1e-6
    return hit, len(exp_docs)


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(out_dir, raw):
    """Writes one step's results, the arrays execute_batch_arrays returns, as out_dir/<name>.npy so that
    two builds can be compared output for output: doc_ids [B, limit] (float64: ids < 2**53 are exact),
    scores [B, limit] float32, n [B] and count [B] float64.  Slots past n hold the library's padding (0).
    When the whole batch exceeds DUMP_CAP_BYTES, a fixed seeded sample of its queries is written and
    query_index [b] (float64) names the rows kept."""
    docs, scores, n, cnt = raw
    B, limit = docs.shape
    per_query = limit * (8 + 4) + 8 + 8 + 8
    room = DUMP_CAP_BYTES - 5 * 128          # five .npy headers of 128 bytes
    rows = np.arange(B)
    if B * per_query > room:
        rows = np.sort(np.random.default_rng(0).choice(B, room // per_query, replace=False))
    out = {"doc_ids": docs[rows].astype(np.float64), "scores": scores[rows].astype(np.float32),
           "n": n[rows].astype(np.float64), "count": cnt[rows].astype(np.float64)}
    if rows.size < B:
        out["query_index"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    args = parse()
    w = dict(WORKLOADS[args.workload])
    batch = args.batch or w["batch"]
    n_docs = args.n_docs or w["n_docs"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank == 0:
            run_reference(args, w, batch, n_docs)
        return

    import torch
    import torch.distributed as dist
    import oramacore_b200 as ob

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = ob.Context(local_rank)
    if world > 1:
        uid = [ob.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(world, rank, uid[0])
        if os.environ.get("OC_SHARD_P2P", "1") != "0":   # direct NVLink exchange of the shard records (else ncclAllGather)
            def _ag(blob):
                out = [None] * world
                dist.all_gather_object(out, blob)
                return out
            ctx.comm_enable_p2p(_ag)

    check = not args.no_cpu_baseline
    wl = make_workload(w, n_docs, batch, rank, world, keep_all=(rank == 0 and check))
    lo, hi = wl["lo"], wl["hi"]
    emb = strs = None
    if w["dim"]:
        emb = ob.EmbeddingFieldStorage(ctx, dim=w["dim"], model="BGEBase" if w["dim"] == 768 else "BGELarge",
                                       dtype=w.get("dtype", "f32"))
        emb.reserve(hi - lo)
        ids = np.arange(lo, hi, dtype=np.uint64)
        if wl.get("chunked"):
            from oramacore_b200 import synth
            CH = 1 << 18
            for c0 in range(0, n_docs, CH):        # chunk c uses seed SEED+c (chunk 0 == the planted chunk)
                c1 = min(n_docs, c0 + CH)
                a, b = max(c0, lo), min(c1, hi)
                if a >= b:
                    continue
                chunk = synth.make_vectors(c1 - c0, w["dim"], seed=synth.SEED_VECTORS + (c0 // CH) * (c0 > 0))
                emb.insert_batch(np.arange(a, b, dtype=np.uint64), chunk[a - c0:b - c0])
        else:
            for i in range(0, hi - lo, 1 << 18):
                emb.insert_batch(ids[i:i + (1 << 18)], wl["rows"][i:i + (1 << 18)])
    if w["vocab"]:
        if world == 1:
            strs = ob.StringFieldStorage(ctx, wl["data_all"])
        else:
            from oramacore_b200.sharding import shard_string_index
            sd, gdf = shard_string_index(wl["data_all"], lo, hi)
            strs = ob.StringFieldStorage(ctx, sd, global_df=gdf)
    mode = {"fulltext": ob.MODE_FULLTEXT, "vector": ob.MODE_VECTOR, "hybrid": ob.MODE_HYBRID}[w["mode"]]
    tsc = ob.TokenScoreContext(ctx, emb, strs)
    params = ob.TokenScoreParams(mode=mode, limit_hint=10, similarity=0.0, sharded=world > 1)
    texts = wl.get("texts")
    qv = wl.get("qv")
    # the step's inputs as they sit in host memory: resolved term ids (packed CSR) + query vectors (pinned)
    packed = [ob.TextQueryBatch(t) for t in texts] if texts is not None else [None] * N_BATCHES
    qv_host = [None] * N_BATCHES
    if qv is not None:
        for i in range(N_BATCHES):
            qv_host[i] = ob.pinned_empty(qv[i].shape, np.float32)
            qv_host[i][...] = qv[i]

    def step(k):
        return tsc.execute_batch_arrays(params, packed[k % N_BATCHES], qv_host[k % N_BATCHES])

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    n_warm = max(args.warmup, 3)
    for k in range(n_warm):
        step(k)
    launches0 = ctx.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    acc = dict(device_ms=0.0, scan_ms=0.0, bm25_ms=0.0, fuse_ms=0.0, comm_ms=0.0, scan_sweep_ms=0.0, scan_bytes=0,
               scan_launches=0, bm25_postings=0, scan_unproven=0, scan_rescored=0, rerun_ms=0.0)
    h2d = d2h = tensor_core = variant = 0
    last = [None] * N_BATCHES
    sync_all()
    t0 = time.perf_counter()
    for k in range(args.steps):
        last[k % N_BATCHES] = step(k)
        t = ctx.last_timing()
        for key in acc:
            acc[key] += t.get(key, 0)
        h2d, d2h = t["h2d_bytes"], t["d2h_bytes"]
        tensor_core = max(tensor_core, t["scan_tensor_core"]); variant = max(variant, t["scan_variant"])
    sync_all()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launch_count() - launches0
    for nb in range(N_BATCHES):          # batches the timed loop did not reach (steps < N_BATCHES)
        if last[nb] is None:
            last[nb] = step(nb)

    dev_ms, scan_ms, bm_ms, fuse_ms, comm_ms, sweep_ms = (acc[k] for k in ("device_ms", "scan_ms", "bm25_ms", "fuse_ms", "comm_ms", "scan_sweep_ms"))
    ranks_agree = None
    if world > 1:
        red = torch.tensor([dev_ms, wall * 1e3, scan_ms, bm_ms, fuse_ms, comm_ms, sweep_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(red, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms, scan_ms, bm_ms, fuse_ms, comm_ms, sweep_ms = red.tolist()
        tot = torch.tensor([float(launches)], device="cuda", dtype=torch.float64)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        launches = int(tot.item())
        # every rank holds the global answer after the all-gather merge: they must be byte-identical
        h = hashlib.sha1()
        for r in last:
            for a in r:
                h.update(np.ascontiguousarray(a).tobytes())
        digests = [None] * world
        dist.all_gather_object(digests, h.hexdigest())
        ranks_agree = len(set(digests)) == 1
    else:
        wall_ms = wall * 1e3
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    K, B = args.steps, batch
    if args.dump_outputs:      # every rank holds the merged answer: rank 0 writes it
        dump_outputs(args.dump_outputs, last[(K - 1) % N_BATCHES])
    value = B * K / (dev_ms * 1e-3)
    e2e = B * K / (wall_ms * 1e-3)
    pk, peak_src = peaks()
    peak = float(pk["hbm_gbs"])
    cfg = config_of(w, B, n_docs)
    cfg.update({"parallelism": f"doc-shard x{world}", "l2_flush": "inputs larger than L2 (matrix >> 126 MB)"})
    line = {
        "metric": METRIC.get(args.workload, f"{w['mode']}_search_qps"),
        "value": value, "unit": "queries/s", "n_gpus": world, "steps": K, "warmup": n_warm,
        "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "bf16 storage, f32 arithmetic" if w.get("dtype") == "bf16" else "f32", "data": "synthetic",
        "config": cfg,
        "e2e": {"value": e2e, "unit": "queries/s", "ms_per_step": wall_ms / K, "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h)},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "stage_ms_per_step": {"scan": scan_ms / K, "scan_sweep_kernel": sweep_ms / K, "bm25": bm_ms / K, "fuse": fuse_ms / K, "comm": comm_ms / K},
    }
    # roofline of the dominant kernel
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(args.workload)
    scan_bytes, scan_launches, postings = acc["scan_bytes"], acc["scan_launches"], acc["bm25_postings"]
    if w["dim"]:   # vector / hybrid: the matrix sweep is the dominant kernel (the fulltext stage overlaps it on the side stream)
        # dominant kernel = the sweep launch(es): CUDA events around those launches on the library's stream
        # (scan stage = threshold pass + sweep; its fraction is reported as batch_level_frac)
        ach = (scan_bytes / 1e9) / (max(sweep_ms, 1e-9) * 1e-3)
        n_local = hi - lo
        tflops = (2.0 * B * n_local * w["dim"] / 1e12) / (max(sweep_ms, 1e-9) / K * 1e-3) if tensor_core else None
        kname, kdesc = SCAN_VARIANTS.get(variant, ("emb_scan_kernel", "exact fp32 sweep"))
        line["scan"] = {"kernel": f"{kname} ({kdesc})",
                        "queries_rerun_through_exact_sweep_per_step": acc["scan_unproven"] / K,
                        "rerun_ms_per_step": acc["rerun_ms"] / K,
                        "rows_rescored_exactly_per_query": acc["scan_rescored"] / K,
                        "tensor_tflops_per_gpu": tflops}
        if tensor_core and w.get("dtype") == "bf16" and B >= 512:
            tpeak = float(pk.get("bf16_tflops_sustained", 1400.0))
            line["roofline_tensor"] = {"kernel": kname, "bound": "tensor", "achieved": tflops, "peak": tpeak,
                                       "unit": "TFLOP/s", "frac": tflops / tpeak,
                                       "peak_source": f"of {peak_src} (sustained)"}
        line["roofline"] = {"kernel": kname, "bound": "hbm", "achieved": ach, "peak": peak,
                            "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "peak_source": f"of {peak_src}",
                            "kernel_ms_per_launch": sweep_ms / max(scan_launches, 1), "launches_per_step": scan_launches / K,
                            "algorithmic_bytes_per_launch": scan_bytes / max(scan_launches, 1),
                            "batch_level_frac": (scan_bytes / max(scan_launches, 1) * K / 1e9) / (scan_ms * 1e-3) / peak}
    else:
        ach = (postings * 8 / 1e9) / (bm_ms * 1e-3)
        line["roofline"] = {"kernel": "bm25_warp_kernel (whole fulltext stage timed: plan + precompute + seed + scorer)", "bound": "hbm", "achieved": ach, "peak": peak,
                            "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "peak_source": f"of {peak_src}",
                            "postings_per_s": postings / (bm_ms * 1e-3)}
    if w["dim"] and w["vocab"] and postings:
        line["roofline_bm25"] = {"kernel": "bm25_warp_kernel (whole fulltext stage timed)", "bound": "hbm", "achieved": (postings * 8 / 1e9) / (bm_ms * 1e-3),
                                 "peak": peak, "unit": "GB/s", "frac": (postings * 8 / 1e9) / (bm_ms * 1e-3) / peak,
                                 "postings_per_s": postings / (bm_ms * 1e-3), "stage_ms": bm_ms / K,
                                 "note": "the fulltext stage runs on the side stream under the matrix sweep: its window includes the wait for "
                                         "the SMs' shared memory the sweep holds (OC_SIDE_STREAM=0 times it alone: profiles/)"}

    def hits_of(raw, i):
        return ob.SearchHits(raw[0][i, :raw[2][i]].copy(), raw[1][i, :raw[2][i]].copy(), int(raw[3][i]))

    # ---- parity / recall of the timed configuration + CPU baseline (outside the timed region)
    if wl.get("chunked"):
        hp = sum(int(last[nb][0][i, 0]) == int(wl["planted"][nb][i]) for nb in range(N_BATCHES) for i in range(B))
        line["parity"] = {"planted_neighbour_is_rank1": hp, "queries": B * N_BATCHES, "ranks_agree": ranks_agree,
                          "note": "corpus generated chunk-wise (41 GB in fp32): no host copy for the CPU oracle; parity of this path is covered by tests/test_gpu_gemm.py::test_bf16_store_parity"}
    elif check:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle as orc
        rows_all = wl.get("rows_all")
        ix = orc.StrIndex(wl["data_all"]) if w["vocab"] else None
        st = orc.EmbStore(rows_all) if w["dim"] else None
        cores = os.cpu_count() or 1
        # round-robin over the rotated batches: every batch is sampled
        order = [(nb, i) for i in range(B) for nb in range(N_BATCHES)]
        done, tcpu, agree, rh, rt = 0, 0.0, 0, 0, 0
        while done < len(order) and tcpu < args.cpu_seconds:
            chunk = order[done:done + cores]
            sb = orc.SearchBatch(ix, st)
            for nb, i in chunk:
                sb.add(mode, limit=10, similarity=0.0, q_vec=qv[nb][i] if w["dim"] else None,
                       text=texts[nb][i] if w["vocab"] else None)
            t1 = time.perf_counter()
            od, os_, on, oc = sb.run(cores)
            tcpu += time.perf_counter() - t1
            for k, (nb, i) in enumerate(chunk):
                h = hits_of(last[nb], i)
                exp = set(od[k, :on[k]].tolist())
                agree += (set(h.doc_ids.tolist()) == exp and h.count == int(oc[k])
                          and h.scores.shape[0] == int(on[k]) and np.allclose(h.scores, os_[k, :on[k]], atol=1e-5, rtol=0))
                rt += len(exp)
                rh += len(exp & set(h.doc_ids.tolist()))
            done += len(chunk)
        line["cpu_baseline"] = {"value": done / tcpu, "unit": "queries/s", "cores": cores, "kind": "port",
                                "sample": f"{done} of the {B * N_BATCHES} timed queries (round-robin over the {N_BATCHES} batches), one query per "
                                          f"thread, {tcpu:.1f} s of CPU work; C restatement of the reference algorithm "
                                          "(per-query brute-force scan + hash-map BM25), not the Rust binary"}
        line["parity"] = {"queries_checked": done, "identical_to_oracle": int(agree),
                          "recall_at_10_vs_oracle": rh / max(rt, 1), "n_gpus": world, "ranks_agree": ranks_agree,
                          "oracle_corpus": "unsharded"}
        # ---- recall@10 vs fp64 on >= 1000 of the timed queries (SURVEY §8d)
        if w["dim"] and args.recall_queries:
            nq = min(args.recall_queries, B * N_BATCHES)
            pick = order[:nq]
            t1 = time.perf_counter()
            Q = np.stack([qv[nb][i] for nb, i in pick])
            vi, vs = fp64_vector_topk(rows_all, Q, 10)
            hit = tot = 0
            if w["mode"] == "hybrid":
                from concurrent.futures import ThreadPoolExecutor

                tl = threading.local()

                def one(k):
                    nb, i = pick[k]
                    if not hasattr(tl, "buf"):
                        tl.buf = np.zeros(n_docs)
                    ed, es = fp64_hybrid_topk(wl["data_all"], texts[nb][i], vi[k], vs[k], 10, scratch=tl.buf)
                    h = hits_of(last[nb], i)
                    return recall_hits(h.doc_ids, ed, es, h.scores)
                with ThreadPoolExecutor(min(32, cores)) as ex:
                    for a, b in ex.map(one, range(nq)):
                        hit += a; tot += b
            else:
                for k, (nb, i) in enumerate(pick):
                    h = hits_of(last[nb], i)
                    a, b = recall_hits(h.doc_ids, vi[k].tolist(), vs[k].tolist(), h.scores)
                    hit += a; tot += b
            line["parity"]["recall_at_10_vs_fp64"] = hit / max(tot, 1)
            line["parity"]["recall_queries"] = nq
            line["parity"]["recall_seconds"] = round(time.perf_counter() - t1, 1)

    # ---- driver-visible sub-result for BASELINE configs[1]: B = 1 scan on the resident matrix
    if args.workload == "h1" and world == 1 and not args.no_extra:
        vp = ob.TokenScoreParams(mode=ob.MODE_VECTOR, limit_hint=10, similarity=0.0)
        nq1 = min(32, B * N_BATCHES)
        q1 = ob.pinned_empty((nq1, 1, w["dim"]), np.float32)
        for k in range(nq1):
            q1[k, 0] = qv[k % N_BATCHES][k // N_BATCHES]
        for k in range(3):
            tsc.execute_batch_arrays(vp, None, q1[k])
        K1 = 20
        d1 = s1 = 0.0
        b1 = l1 = 0
        res1 = []
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        for k in range(K1):
            res1.append(tsc.execute_batch_arrays(vp, None, q1[(3 + k) % nq1]))
            t = ctx.last_timing()
            d1 += t["device_ms"]; s1 += t["scan_sweep_ms"]; b1 += t["scan_bytes"]; l1 += t["scan_launches"]
        torch.cuda.synchronize()
        w1 = (time.perf_counter() - t1) * 1e3
        ach1 = (b1 / 1e9) / (s1 * 1e-3)
        ex = {"config": WORKLOADS["v1"]["desc"], "value": K1 / (d1 * 1e-3), "unit": "queries/s", "steps": K1,
              "ms_per_step": d1 / K1, "e2e": {"value": K1 / (w1 * 1e-3), "unit": "queries/s", "ms_per_step": w1 / K1},
              "roofline": {"kernel": "emb_scan_kernel", "bound": "hbm", "achieved": ach1, "peak": peak, "unit": "GB/s",
                           "frac": ach1 / peak, "kernel_ms_per_launch": s1 / max(l1, 1),
                           "algorithmic_bytes_per_launch": b1 / max(l1, 1), "peak_source": f"of {peak_src}"}}
        if check:
            ok = 0
            for k in range(K1):
                od, os_ = orc.vector(st, q1[(3 + k) % nq1, 0], 10, 0.0)
                o = np.argsort(-os_, kind="stable")
                r = res1[k]
                ok += (set(r[0][0, :r[2][0]].tolist()) == set(od.tolist())
                       and np.allclose(r[1][0, :r[2][0]], os_[o], atol=1e-5, rtol=0))
            ex["parity"] = {"queries_checked": K1, "identical_to_oracle": int(ok)}
        line["extra"] = {"v1": ex}
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
