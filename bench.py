#!/usr/bin/env python
"""bench.py -- BM25 queries/s of the batched posting-traversal path (BASELINE.json configs[1]):
10M-doc synthetic Zipf corpus, 1024 three-term disjunctive queries, top-100, on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload bm25|conj|knn|hybrid] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over the 1024-query batch. `value` = whole-job queries/s with the compiled batch
resident in HBM; `e2e` = the same through the public one-shot call with HOST query buffers (query upload + result
download inside the timed region). N > 1: the corpus is split into N contiguous doc-range shards (one per GPU, index-wide
BM25 statistics all-reduced at build time); every step ends with ONE NCCL all-gather of the packed per-shard results
(docs, scores, counts, relation flags, totalHits) and a device-side TopDocs.merge => strong scaling.

Every number is gated: before timing, the results of the first `--cpu-sample` queries are compared bit for bit with the CPU
oracle (at N > 1 the MERGED page against the oracle run on the whole corpus by rank 0). The default N = 1 line also carries
`extra.conj` (configs[2]) and `extra.knn` (configs[3]), each with its own gate and roofline.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("NRT_ORACLE_NATIVE", "1")   # the CPU baseline is the oracle compiled -O3 -march=native ON THE BOX THAT RUNS IT

ALG_BYTES_PER_POSTING = 9  # SURVEY.md 8d: int32 doc id + int32 freq + 1 B norm gather
INT_MAX = 2**31 - 1


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--docs", type=int, default=10_000_000)
    ap.add_argument("--vocab", type=int, default=1_000_000)
    ap.add_argument("--nq", type=int, default=1024)
    ap.add_argument("--topk", type=int, default=100)
    ap.add_argument("--threshold", type=int, default=1000, help="totalHitsThreshold (reference default 1000)")
    ap.add_argument("--cpu-sample", type=int, default=1024, help="queries in the bounded CPU-baseline / gate sample")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[2] / configs[3] legs of the default N=1 line")
    ap.add_argument("--workload", default="bm25", choices=["bm25", "conj", "knn", "hybrid"],
                    help="bm25 = configs[1] (the headline line); conj = configs[2]; knn = configs[3] (1..8 GPUs); hybrid = configs[4] shape")
    ap.add_argument("--hybrid-docs-per-gpu", type=int, default=12_500_000, help="--workload hybrid: docs (text + one vector each) per GPU")
    ap.add_argument("--hybrid-dims", type=int, default=128)
    ap.add_argument("--vectors", type=int, default=1_000_000)
    ap.add_argument("--dims", type=int, default=768)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (docs, scores, counts, ...) as DIR/<name>.npy in float32 / float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 60_000_000   # all files together stay below 64 MB, .npy headers included


def dump_outputs(out_dir, arrays):
    """Writes {name: array} with the query as the first axis. Integer arrays become float64 (exact for the doc ids,
    counts and totals here), float32 stays float32. Above DUMP_LIMIT_BYTES a fixed seeded sample of query rows is written,
    with their indices as query_rows.npy, so that two builds run with the same arguments write comparable files."""
    arrays = {name: np.asarray(a, np.float32 if np.asarray(a).dtype == np.float32 else np.float64) for name, a in arrays.items()}
    nq = len(next(iter(arrays.values())))
    row_bytes = sum(a.nbytes // nq for a in arrays.values()) + 8
    if nq * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(nq, DUMP_LIMIT_BYTES // row_bytes, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["query_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def static_traffic(name):
    """Physical DRAM bytes per launch from the committed ncu --set full capture of this exact workload (a STATIC figure:
    the bench cannot run under the profiler). Returns (bytes, source) or (None, None)."""
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))[name]
        return tr["dram_bytes_read"] + tr["dram_bytes_write"], "static: profiles/r2_traffic.json (%s)" % tr["source"]
    except Exception:
        return None, None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (rows are time-stamped on arrival;
    mark() brackets the region)."""

    def __init__(self, device):
        self.rows, self.proc, self.device, self.t0, self.t1 = [], None, device, None, None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
                                         bufsize=1)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def ready(self):
        return self.proc is None or len(self.rows) > 0

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc:
            time.sleep(0.05)
            self.proc.terminate()
        t0 = self.t0 or 0.0
        t1 = self.t1 or time.time()
        inside = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.03]
        if not inside and self.rows:   # region shorter than one sampling period: take the sample closest to it
            inside = [min(self.rows, key=lambda x: abs(x[0] - 0.5 * (t0 + t1)))[1]]
        sm, mx, reasons = [], 0, set()
        for r in inside:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- workloads

def make_queries(nq, vocab):
    from nrtsearch_b200 import index as ix
    from nrtsearch_b200.search import BooleanQuery, Occur, TermQuery
    terms = ix.synth_query_terms(nq, 3, vocab)   # rank log-uniform in [10, 10^4)
    return [BooleanQuery().add(TermQuery(int(t[0])), Occur.SHOULD).add(TermQuery(int(t[1])), Occur.SHOULD)
            .add(TermQuery(int(t[2])), Occur.SHOULD) for t in terms]


def make_conj_queries(nq, vocab, with_filter=True):
    """configs[2]: 2 MUST terms + FILTER price in [lo, lo + 1e5] (10 % selective), SURVEY.md App. B."""
    from nrtsearch_b200 import index as ix
    from nrtsearch_b200.search import BooleanQuery, Occur, RangeQuery, TermQuery
    terms = ix.synth_query_terms(nq, 2, vocab)
    los = (ix.synth_uniform(nq, ix.SEED_RANGE) * 900_000).astype(np.int64)
    qs = []
    for t, lo in zip(terms, los):
        q = BooleanQuery().add(TermQuery(int(t[0])), Occur.MUST).add(TermQuery(int(t[1])), Occur.MUST)
        if with_filter:
            q.add(RangeQuery(0, int(lo), int(lo) + 100_000), Occur.FILTER)
        qs.append(q)
    return qs


def build_shard(args, rank, world, with_column=True):
    """Rank r holds docs [r*N/G, (r+1)*N/G); df / docCount / sumTotalTermFreq become index-wide."""
    from nrtsearch_b200 import index as ix
    from nrtsearch_b200.shards import install_global_stats, shard_range
    lo, hi = shard_range(args.docs, rank, world)
    sh = ix.synth_text_shard(hi - lo, args.vocab, doc_begin=lo)
    if with_column:
        sh.columns = [ix.synth_int_column(hi - lo, doc_begin=lo)]
        sh.column_has = [None]
    if world > 1:
        import torch
        install_global_stats(sh, device=torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))))   # NCCL all-reduce, build time
    else:
        sh.term_df = np.diff(sh.term_off).astype(np.int64)
    return sh


def oracle_run(sh, queries, topk, threshold, mode, threads, repeat=1):
    """The reference's CPU path restated (oracle/): mode 1 = MAXSCORE dynamic pruning for pure disjunctions, one query
    per thread. Returns (queries/s of the last run, results, OracleIndex)."""
    import oracle
    from nrtsearch_b200.search import compile_queries
    oix = oracle.OracleIndex(sh, with_impacts=True)
    carr, ncl, qarr, nq = compile_queries(queries)
    oracle.search_compiled(oix, carr, ncl, qarr, min(nq, 8), topk, threshold, mode, threads)  # warm
    for _ in range(repeat):
        t0 = time.perf_counter()
        res = oracle.search_compiled(oix, carr, ncl, qarr, nq, topk, threshold, mode, threads)
        dt = time.perf_counter() - t0
    return nq / dt, res, oix


def gate(what, got_docs, got_scores, got_counts, ref):
    """Bit-exact doc ids + scores of the sampled queries vs the oracle; raises on any difference."""
    n = len(ref[2])
    assert np.array_equal(got_counts[:n], ref[2]), f"bench gate ({what}): hit counts differ from the CPU oracle"
    for q in range(n):
        c = int(ref[2][q])
        assert np.array_equal(got_docs[q, :c], ref[0][q, :c]), f"bench gate ({what}): top-k doc ids of query {q} differ from the CPU oracle"
        assert np.array_equal(got_scores[q, :c].view(np.uint32), ref[1][q, :c].view(np.uint32)), \
            f"bench gate ({what}): scores of query {q} differ from the CPU oracle"
    return {"queries": n, "bit_exact": True}


def time_batch(batch, stream, steps, warmup=3):
    """Kernel (stage 0) and merge (stage 1) time per run of a prepared batch, CUDA events on the launch stream."""
    import torch
    for _ in range(warmup):
        batch.run(stream)
    torch.cuda.synchronize()
    batch.reset_timing()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        batch.run(stream)
    e1.record()
    torch.cuda.synchronize()
    return batch.stage_ms(0), batch.stage_ms(1), e0.elapsed_time(e1) / steps


def workload_config(args, kind="bm25"):
    if kind == "conj":
        return {"workload": "configs[2]: 10M-doc synthetic, conjunctive AND (2 MUST terms) + int range FILTER, 1024-query batch top-100",
                "docs": args.docs, "vocab": args.vocab, "batch": args.nq, "top_k": args.topk, "sharding": f"doc-range x{args.gpus}"}
    return {"workload": "configs[1]: 10M-doc synthetic Zipf postings, 1024-query disjunctive BM25 top-100",
            "docs": args.docs, "vocab": args.vocab, "batch": args.nq, "terms_per_query": 3, "top_k": args.topk,
            "total_hits_threshold": args.threshold, "sharding": f"doc-range x{args.gpus}",
            "l2": "posting image (GBs) >> 126 MB L2; no flush needed"}


# ---------------------------------------------------------------------------------------------- conj leg (configs[2])

def conj_leg(args, searcher, sh, stream, steps, threads, n_sample):
    """configs[2] on the resident index: gate vs the exhaustive oracle, kernel time, SURVEY 8d byte formula
    sum_q [ sum_t df(t) * 8 B + |intersection_q| * (T + 4) B ]."""
    import torch
    from nrtsearch_b200.search import RelevanceCollector
    queries = make_conj_queries(args.nq, args.vocab)
    coll = RelevanceCollector(args.topk, args.threshold)
    qps_cpu, ref, _ = oracle_run(sh, queries[:n_sample], args.topk, args.threshold, 1, threads)
    res = searcher.search_batch(queries, coll)
    g = gate("conj", res.docs, res.scores, res.counts, ref)
    # |intersection|: the same conjunctions without the range filter, exact counts
    inter = searcher.search_batch(make_conj_queries(args.nq, args.vocab, with_filter=False), RelevanceCollector(1, INT_MAX)).total_hits
    batch = searcher.prepare(queries, coll)
    stats = batch.stats()
    kernel_ms, merge_ms, step_ms = time_batch(batch, stream, steps)
    batch.close()
    # e2e: the one-shot C-ABI call with HOST query buffers (compiled once, as a serving adaptor would cache them) and host results
    from nrtsearch_b200.search import compile_queries
    from nrtsearch_b200 import _native
    carr, ncl, qarr, _ = compile_queries(queries)
    hd, hs = np.zeros((args.nq, args.topk), np.int32), np.zeros((args.nq, args.topk), np.float32)
    hc, ht, hr = np.zeros(args.nq, np.int32), np.zeros(args.nq, np.int64), np.zeros(args.nq, np.uint8)
    lib = _native.gpu_lib()

    def e2e_call():
        _native.check(lib.nrtgpu_search_bool(searcher.index.handle, carr, ncl, qarr, args.nq, args.topk, args.threshold, 0, ctypes.c_void_p(stream),
                                             hd.ctypes.data, hs.ctypes.data, hc.ctypes.data, ht.ctypes.data, hr.ctypes.data))
    for _ in range(2):
        e2e_call()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_call()
    e2e = args.nq * steps / (time.perf_counter() - t0)
    assert np.array_equal(hd[:len(ref[2])][:, :1], res.docs[:len(ref[2])][:, :1]), "bench (conj): the one-shot call disagrees with the prepared batch"
    pk, src = peaks()
    alg = float(stats["alg_postings"]) * 8.0 + float(inter.sum()) * (2 + 4) + args.nq * args.topk * 8
    ach = alg / (kernel_ms * 1e-3) / 1e9
    return {"metric": "conjunctive (2 MUST + range FILTER) queries/sec (batch 1024, 10M docs)", "value": args.nq / (step_ms * 1e-3),
            "unit": "queries/s", "ms_per_step": step_ms, "config": workload_config(args, "conj"),
            "e2e": {"value": e2e, "unit": "queries/s"}, "gate": g,
            "roofline": {"bound": "hbm", "kernel": "posting_probe_kernel<generic> (leap-frog: the rarest MUST list leads, the other list is probed, norm / doc-value gathers only for the intersection)",
                         "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "peak_source": src,
                         "kernel_ms": kernel_ms, "merge_ms": merge_ms, "alg_bytes_per_launch": alg,
                         "alg_formula": "sum_q [sum_t df(t) * 8 B + |intersection_q| * (2 + 4) B] + nq * k * 8 B (SURVEY.md 8d)",
                         "intersection_docs": int(inter.sum())},
            "cpu_baseline": {"value": qps_cpu, "unit": "queries/s", "cores": threads, "kind": "port",
                             "sample": f"first {n_sample} queries, exhaustive DAAT (oracle/oracle.c), same corpus"}}


# ---------------------------------------------------------------------------------------------- kNN (configs[3])

def knn_leg(args, rank, world, local_rank, steps, warmup, outputs=None):
    """configs[3]: 1M x 768 fp32 vectors, batch-1024 cosine top-100; exact search (tcgen05 bf16 candidate stage, fp64
    re-score, rank-safety certificate). world > 1: the corpus is row-partitioned, every rank searches its shard, ONE
    all-gather of the packed results, TopDocs.merge on the device. `outputs` (a dict) receives the page of the last
    timed step."""
    import torch
    import oracle
    from nrtsearch_b200 import _native, index as ix
    from nrtsearch_b200.index import HostShard
    from nrtsearch_b200.search import GpuContext, GpuIndex
    from nrtsearch_b200.shards import PackedGather, shard_range
    n, dims, nq, k = args.vectors, args.dims, args.nq, args.topk
    lo, hi = shard_range(n, rank, world)
    corpus = ix.synth_vectors(hi - lo, dims, row_begin=lo)
    queries = ix.synth_vectors(nq, dims, seed=ix.SEED_VQUERIES)
    sh = HostShard(n_docs=hi - lo, doc_base=lo, term_off=np.zeros(1, np.int64), post_docs=np.zeros(0, np.int32),
                   post_freqs=np.zeros(0, np.int32), fields=[], vectors=corpus, vec_similarity=ix.SIM_COSINE)
    ctx = GpuContext(local_rank)
    gix = GpuIndex(ctx, sh)
    lib = _native.gpu_lib()
    dev = torch.device("cuda", local_rank)
    docs, scores, counts = np.zeros((nq, k), np.int32), np.zeros((nq, k), np.float32), np.zeros(nq, np.int32)
    stage = (ctypes.c_float * 3)()
    stream = torch.cuda.current_stream().cuda_stream
    pg = PackedGather(nq, k, world, dev) if world > 1 else None
    host_rec = torch.zeros(pg.words, dtype=torch.int32).pin_memory() if pg else None

    def call():
        _native.check(lib.nrtgpu_search_knn_timed(gix.handle, queries.ctypes.data, nq, k, ctypes.c_void_p(stream), docs.ctypes.data,
                                                  scores.ctypes.data, counts.ctypes.data, stage))
        if pg:   # per-shard page -> packed record -> one all-gather -> device merge -> merged page on the host
            r = host_rec.numpy()
            r[:nq * k] = docs.reshape(-1); r[nq * k:2 * nq * k] = scores.reshape(-1).view(np.int32); r[2 * nq * k:2 * nq * k + nq] = counts
            pg.local.copy_(host_rec, non_blocking=True)
            pg.gather(); pg.merge_on_device(ctx, stream)
            return pg.unpack()
        return docs, scores, counts, None, None

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(warmup, 1)):
        out = call()
    uncert = int(lib.nrtgpu_knn_last_uncertified(gix.handle))
    barrier()
    gemm, sel, resc = [], [], []
    sampler.mark_begin()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = call()
        gemm.append(stage[0]); sel.append(stage[1]); resc.append(stage[2])
    barrier()
    wall = (time.perf_counter() - t0) / steps
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    if outputs is not None:
        outputs.update(docs=out[0].copy(), scores=out[1].copy(), counts=out[2].copy())
    dev_ms = float(np.mean(gemm) + np.mean(sel) + np.mean(resc))
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([wall, dev_ms, float(np.mean(gemm))], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall, dev_ms, gemm_ms = float(t[0]), float(t[1]), float(t[2])
    else:
        gemm_ms = float(np.mean(gemm))
    line = None
    if rank == 0:
        threads = os.cpu_count() or 1
        whole = corpus if world == 1 else ix.synth_vectors(n, dims)
        ns = min(32, nq)
        t0 = time.perf_counter()
        wd, ws, wc = oracle.knn_exact(whole, ix.SIM_COSINE, queries[:ns], k, n_threads=threads)
        cpu_qps = ns / (time.perf_counter() - t0)
        gd, gs = out[0], out[1]
        recall = float(np.mean([len(set(gd[q]) & set(wd[q])) / k for q in range(ns)]))
        bad = [q for q in range(ns) if not np.array_equal(gd[q], wd[q])]
        for q in bad:   # ids may differ only inside a score tie band (1e-5 relative), as in tests/test_gpu_knn.py
            np.testing.assert_allclose(np.sort(gs[q])[::-1], ws[q], rtol=1e-5)
            assert set(gd[q]) == set(wd[q]) or abs(gs[q, -1] - ws[q, -1]) <= 1e-5 * abs(ws[q, -1]), "bench gate (knn): ids differ from the exact oracle"
        np.testing.assert_allclose(gs[:ns], ws, rtol=1e-5, err_msg="bench gate (knn): scores differ from the exact oracle")
        pk, src = peaks()
        flops = 2.0 * nq * n * dims
        ach = flops / world / (gemm_ms * 1e-3) / 1e12   # per GPU: every rank multiplies the batch by its 1/world of the corpus
        line = {"metric": "kNN queries/sec (batch 1024, 1M x 768 cosine top-100, exact)", "value": nq / (dev_ms * 1e-3) if world == 1 else nq / wall,
                "unit": "queries/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": dev_ms if world == 1 else wall * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16 candidates + f64 exact re-score",
                "data": "synthetic",
                "config": {"workload": "configs[3]: 1M x 768-d fp32 vectors, batch-1024 cosine top-100", "vectors": n, "dims": dims, "batch": nq,
                           "top_k": k, "sharding": f"row-partition x{world}"},
                "e2e": {"value": nq / wall, "unit": "queries/s", "h2d_bytes_per_step": nq * dims * 4, "d2h_bytes_per_step": nq * k * 8 + nq * 4},
                "recall_at_k_vs_exact": recall,
                "gate": {"queries": ns, "ids_equal_oracle": ns - len(bad), "tie_band_only": len(bad), "scores_rtol": 1e-5},
                "certificate": {"uncertified_queries": uncert, "of": nq,
                                "rule": "every vector outside the k' = 4k candidate list proven below the k-th exact score with the bf16 error bound 2^-7 |q||d|; rejected queries re-run exactly"},
                "roofline": {"bound": "tensor", "kernel": "knn_gemm_bf16_db_kernel (tcgen05 UMMA, 256x128 tiles double-buffered in TMEM, TMA operand ring, 16 epilogue warps with the fused top-k' threshold filter)",
                             "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"], "traffic": None,
                             "peak_source": src + " burst", "gemm_ms": gemm_ms, "select_ms": float(np.mean(sel)), "rescore_ms": float(np.mean(resc))},
                "cpu_baseline": {"value": cpu_qps, "unit": "queries/s", "cores": threads, "kind": "port",
                                 "sample": f"{ns} queries, exact fp64 brute force (oracle/oracle.c), same corpus"},
                "clocks": clocks}
    gix.close(); ctx.close()
    return line


def run_hybrid(args, rank, world, local_rank):
    """configs[4]: docs sharded by doc range over the GPUs (12.5M docs x 128-d per GPU by default = 100M docs at 8 GPUs), every
    shard runs the text retriever (3-term disjunction, top-100, index-wide statistics) and the kNN retriever (cosine,
    k = 100); ONE all-gather moves both packed per-shard pages, every rank merges each retriever's pages (TopDocs.merge)
    and blends them with weighted RRF (rankConstant 60, boosts 1; BlenderOperation.java:76-87). Everything goes through
    the C ABI; the gate is a DISTRIBUTED oracle: each rank's host computes its shard's exact pages (oracle/oracle.c),
    rank 0 merges and blends them on the CPU and compares the final page bit for bit."""
    import torch
    import __graft_entry__ as g
    g.build_if_needed()
    import oracle
    from nrtsearch_b200 import _native, index as ix
    from nrtsearch_b200.search import GpuContext, GpuIndex, GpuIndexSearcher, RelevanceCollector, blend_rrf, compile_queries
    from nrtsearch_b200.shards import PackedGather, shard_range, unpack_record
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; nrtsearch_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    per_gpu = args.hybrid_docs_per_gpu
    args.docs = per_gpu * world          # weak scaling: the corpus grows with the GPUs (configs[4] = 100M docs at 8)
    dims, nq, k = args.hybrid_dims, args.nq, args.topk
    lo, hi = shard_range(args.docs, rank, world)
    t_build = time.perf_counter()
    sh = build_shard(args, rank, world, with_column=False)
    sh.vectors = ix.synth_vectors(hi - lo, dims, row_begin=lo)
    sh.vec_similarity = ix.SIM_COSINE
    queries = make_queries(nq, args.vocab)
    qvec = ix.synth_vectors(nq, dims, seed=ix.SEED_VQUERIES)
    ctx = GpuContext(local_rank); gix = GpuIndex(ctx, sh); s = GpuIndexSearcher(gix)
    build_s = time.perf_counter() - t_build
    lib = _native.gpu_lib()
    coll = RelevanceCollector(k, args.threshold)
    batch = s.prepare(queries, coll)
    words = int(lib.nrtgpu_packed_words(nq, k))
    comb = torch.zeros(2 * words, dtype=torch.int32, device=dev)            # [text record | kNN record] of this shard
    allrec = torch.zeros(world * 2 * words, dtype=torch.int32, device=dev)
    text_all = torch.zeros(world * words, dtype=torch.int32, device=dev)
    knn_all = torch.zeros(world * words, dtype=torch.int32, device=dev)
    merged = torch.zeros(2 * words, dtype=torch.int32, device=dev)
    host_rec = torch.zeros(words, dtype=torch.int32).pin_memory()
    host_out = torch.zeros(2 * words, dtype=torch.int32).pin_memory()
    batch.bind_packed(comb.data_ptr())
    stream = torch.cuda.current_stream().cuda_stream
    kd, ks, kc = np.zeros((nq, k), np.int32), np.zeros((nq, k), np.float32), np.zeros(nq, np.int32)

    def step():
        batch.run(stream)                                                   # text page of the shard -> comb[:words] (device)
        _native.check(lib.nrtgpu_search_knn(gix.handle, qvec.ctypes.data, nq, k, None, None, ctypes.c_void_p(stream),
                                            kd.ctypes.data, ks.ctypes.data, kc.ctypes.data))
        r = host_rec.numpy()
        r[:nq * k] = kd.reshape(-1); r[nq * k:2 * nq * k] = ks.reshape(-1).view(np.int32); r[2 * nq * k:2 * nq * k + nq] = kc
        comb[words:].copy_(host_rec, non_blocking=True)
        if world > 1:
            dist.all_gather_into_tensor(allrec, comb)                       # the ONE collective of the step
        else:
            allrec.copy_(comb)
        v = allrec.view(world, 2, words)
        text_all.view(world, words).copy_(v[:, 0, :]); knn_all.view(world, words).copy_(v[:, 1, :])
        _native.check(lib.nrtgpu_merge_topk_packed(ctx.handle, world, nq, k, text_all.data_ptr(), merged.data_ptr(), ctypes.c_void_p(stream)))
        _native.check(lib.nrtgpu_merge_topk_packed(ctx.handle, world, nq, k, knn_all.data_ptr(), merged[words:].data_ptr(), ctypes.c_void_p(stream)))
        host_out.copy_(merged, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        h = host_out.numpy()
        td, ts, tc, _, _ = unpack_record(h[:words], nq, k)
        nd, ns_, nc, _, _ = unpack_record(h[words:], nq, k)
        return blend_rrf(ctx, np.stack([td, nd]), np.stack([tc, nc]), [1.0, 1.0], 60, k), (td, ts, tc), (nd, ns_, nc)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- gate: distributed oracle on the first queries
    ns = 0 if args.no_check else min(8, nq)
    (bd, bs, bc, bt), _, _ = step()
    barrier()
    gate_info = None
    if ns:
        carr, ncl, qarr, _ = compile_queries(queries[:ns])
        threads = max(1, (os.cpu_count() or 1) // world)
        od, os_, oc, _, _ = oracle.search_compiled(oracle.OracleIndex(sh), carr, ncl, qarr, ns, k, INT_MAX, 0, threads)
        xd, xs, xc = oracle.knn_exact(sh.vectors, ix.SIM_COSINE, qvec[:ns], k, n_threads=threads)
        xd = xd + lo                                                        # the oracle's kNN page is shard-local
        mine = (od, os_, oc, xd, xs, xc)
        if world > 1:
            pages = [None] * world
            dist.all_gather_object(pages, mine)
        else:
            pages = [mine]
        if rank == 0:
            same = 0
            for q in range(ns):
                def merge(di, si, ci):   # TopDocs.merge: score desc, doc asc
                    d = np.concatenate([pg_[di][q, :pg_[ci][q]] for pg_ in pages]); sc = np.concatenate([pg_[si][q, :pg_[ci][q]] for pg_ in pages])
                    o = np.lexsort((d, -sc.astype(np.float64)))[:k]
                    return d[o], sc[o]
                tdq, _ = merge(0, 1, 2)
                ndq, _ = merge(3, 4, 5)
                pad = lambda a: np.concatenate([a, np.zeros(k - len(a), a.dtype)])
                wd, ws, wt = oracle.blend_rrf(np.stack([pad(tdq), pad(ndq)]), [len(tdq), len(ndq)], [1.0, 1.0], 60, k)
                ok = np.array_equal(bd[q, :bc[q]], wd) and np.array_equal(bs[q, :bc[q]].view(np.uint32), np.asarray(ws, np.float32).view(np.uint32))
                same += int(ok)
            assert same == ns, f"bench gate (hybrid N={world}): {ns - same} of {ns} blended pages differ from the distributed CPU oracle"
            gate_info = {"queries": ns, "bit_exact": True, "against": "per-shard oracle pages (text: exact BM25, kNN: fp64 brute force) merged and RRF-blended on the CPU"}
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler.mark_begin()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        last = step()
    barrier()
    wall = (time.perf_counter() - t0) / args.steps
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([wall], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall = float(t[0])
    if rank == 0:
        stats = batch.stats()
        print(json.dumps({
            "metric": "hybrid BM25 + kNN + weighted-RRF queries/sec (batch 1024, doc-sharded)", "value": nq / wall, "unit": "queries/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": wall * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 BM25; bf16 candidates + f64 exact re-score (kNN)", "data": "synthetic",
            "config": {"workload": "configs[4]: hybrid BM25 + kNN rescorer/blender, doc-range shards, one all-gather of the packed per-shard pages",
                       "docs": args.docs, "docs_per_gpu": per_gpu, "dims": dims, "vocab": args.vocab, "batch": nq, "top_k": k,
                       "sharding": f"doc-range x{world}", "blend": "weighted RRF, rankConstant 60"},
            "e2e": {"value": nq / wall, "unit": "queries/s", "h2d_bytes_per_step": nq * 3 * 24 + nq * dims * 4 + words * 4,
                    "d2h_bytes_per_step": 2 * words * 4 + nq * k * 8},
            "timing": "host wall clock per step (the step is host-driven: C-ABI calls with host buffers), barrier + synchronize on both sides, max over ranks",
            "gpu_launches": int(stats["launches_per_run"]) + 8, "gate": gate_info, "clocks": clocks,
            "index": {"postings_rank0": int(sh.term_off[-1]), "device_bytes_rank0": gix.device_bytes, "build_s": build_s}}))
        if args.dump_outputs:
            (bd, bs, bc, bt), _, _ = last
            dump_outputs(args.dump_outputs, {"docs": bd, "scores": bs, "counts": bc, "total_hits": bt})
    batch.close(); gix.close(); ctx.close()
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------- reference arm

def run_reference(args, rank, world):
    """The reference's CPU path (restated: oracle/oracle.c, NOT Lucene -- no JVM / lucene-core jar in this image) on all
    host threads, same config / metric; each step = a bounded sample (the first --cpu-sample queries)."""
    if rank != 0:
        return
    import __graft_entry__ as g
    g.build_if_needed()
    threads = os.cpu_count() or 1
    sh = build_shard(args, 0, 1, with_column=args.workload == "conj")
    conj = args.workload == "conj"
    queries = make_conj_queries(args.nq, args.vocab) if conj else make_queries(args.nq, args.vocab)
    n_sample = min(args.cpu_sample, args.nq)
    import oracle
    from nrtsearch_b200.search import compile_queries
    oix = oracle.OracleIndex(sh, with_impacts=True)
    carr, ncl, qarr, nq = compile_queries(queries[:n_sample])
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        res = oracle.search_compiled(oix, carr, ncl, qarr, nq, args.topk, args.threshold, 1, threads)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    dt = float(np.mean(times))
    qps = nq / dt
    sample = f"first {n_sample} of the {args.nq} queries per step, MAXSCORE-pruned DAAT, {threads} threads"
    print(json.dumps({
        "impl": "reference", "metric": "BM25 queries/sec (batch 1024, 10M docs)", "value": qps, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3 * args.nq / n_sample,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.workload),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "restated CPU oracle (oracle/oracle.c, -O3 -march=native), NOT Lucene: no JVM / lucene-core jar exists in this image",
    }))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("docs", "scores", "counts", "total_hits", "relation"), res)))


# ---------------------------------------------------------------------------------------------- main line

def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and os.environ.get("OMP_NUM_THREADS", "1") == "1":   # torchrun pins 1 thread: the corpus generators are OpenMP
        os.environ["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 1) // world))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.workload == "hybrid":
        return run_hybrid(args, rank, world, local_rank)

    import torch
    import __graft_entry__ as g
    g.build_if_needed()
    from nrtsearch_b200 import _native
    from nrtsearch_b200.search import GpuContext, GpuIndex, GpuIndexSearcher, RelevanceCollector, compile_queries
    from nrtsearch_b200.shards import PackedGather, unpack_record

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; nrtsearch_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    if args.workload == "knn":
        outputs = {}
        line = knn_leg(args, rank, world, local_rank, args.steps, args.warmup, outputs)
        if rank == 0:
            print(json.dumps(line))
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, outputs)
        if world > 1:
            dist.destroy_process_group()
        return

    threads = os.cpu_count() or 1
    conj = args.workload == "conj"
    t_build = time.perf_counter()
    sh = build_shard(args, rank, world)
    queries = make_conj_queries(args.nq, args.vocab) if conj else make_queries(args.nq, args.vocab)
    ctx = GpuContext(local_rank)
    gix = GpuIndex(ctx, sh)
    searcher = GpuIndexSearcher(gix)
    coll = RelevanceCollector(args.topk, args.threshold)
    batch = searcher.prepare(queries, coll)
    build_s = time.perf_counter() - t_build
    stats = batch.stats()
    n_postings, dev_bytes = int(sh.term_off[-1]), gix.device_bytes
    nq, k = args.nq, args.topk
    lib = _native.gpu_lib()

    # device buffers (torch = memory + streams + the collective: plumbing only)
    pg = PackedGather(nq, k, world, dev)
    batch.bind_packed(pg.local.data_ptr())
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        batch.run(stream)
        if world > 1:
            pg.gather()                        # ONE exchange step: NCCL all-gather of the packed per-shard results
            pg.merge_on_device(ctx, stream)    # TopDocs.merge on every rank

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- correctness gate before any number is reported: the (merged) page of the first queries vs the CPU oracle
    #      run on the WHOLE corpus (rank 0; bit-exact ids + scores), at every N
    cpu, gate_info = None, None
    n_sample = min(args.cpu_sample, nq)
    step(); barrier()
    if rank == 0:
        whole = sh if world == 1 else build_shard(args, 0, 1)
        qps_cpu, ref, _ = oracle_run(whole, queries[:n_sample], k, args.threshold, 1, threads, repeat=3 if world == 1 else 1)
        if world == 1:
            cpu = {"value": qps_cpu, "unit": "queries/s", "cores": threads, "kind": "port",
                   "sample": f"first {n_sample} of the {nq} queries, %s (oracle/oracle.c, -O3 -march=native), same corpus"
                             % ("exhaustive DAAT" if conj else "MAXSCORE-pruned DAAT, mode 1")}
        if not args.no_check:
            gd, gs, gc, gf, gt = pg.unpack(pg.merged if world > 1 else pg.local)
            gate_info = gate(f"{args.workload} N={world}", gd, gs, gc, ref)
            gate_info["against"] = "oracle on the whole corpus" + (" (merged page after the all-gather)" if world > 1 else "")
        del whole

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step()
    barrier()
    if rank == 0:   # keep the GPU under the same load until the clock sampler delivers (at most ~1.5 s of extra warm-up)
        t_wait = time.time()
        while not sampler.ready() and time.time() - t_wait < 1.5:
            batch.run(stream); torch.cuda.synchronize()
    barrier()
    batch.reset_timing()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_begin()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    # the page of the last timed step, read before the e2e leg below reuses pg.local
    outputs = dict(zip(("docs", "scores", "counts", "relation", "total_hits"), pg.unpack(pg.merged if world > 1 else pg.local))) \
        if rank == 0 and args.dump_outputs else None
    ms = e0.elapsed_time(e1)
    kernel_ms = batch.stage_ms(0)
    merge_ms = batch.stage_ms(1)
    if world > 1:
        t = torch.tensor([ms, kernel_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, kernel_ms = float(t[0]), float(t[1])
        pt = torch.tensor([float(stats["alg_postings"])], device=dev, dtype=torch.float64)
        dist.all_reduce(pt)
        alg_postings_total = float(pt[0])
    else:
        alg_postings_total = float(stats["alg_postings"])
    ms_per_step = ms / args.steps
    qps = nq / (ms_per_step * 1e-3)

    # ---- the same batch with exact counts (ScoreMode.COMPLETE): the exhaustive figure SURVEY.md 8d asks for
    exh_ms = None
    if args.threshold != INT_MAX and not conj:
        bex = searcher.prepare(queries, RelevanceCollector(args.topk, INT_MAX))
        exh_ms, _, _ = time_batch(bex, stream, 5, warmup=2)
        bex.close()
        if world > 1:
            t = torch.tensor([exh_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            exh_ms = float(t[0])

    # ---- e2e: the public one-shot call with HOST query buffers every step: H2D plan, kernels, (all-gather + merge on
    #      the device at N > 1 -- results stay on the device until the merged page), D2H of the final page
    carr, ncl, qarr, _ = compile_queries(queries)
    h2d = ctypes.sizeof(carr) + ctypes.sizeof(qarr)
    d2h = int(pg.words) * 4
    host_rec = torch.zeros(pg.words, dtype=torch.int32).pin_memory()

    def e2e_step():
        _native.check(lib.nrtgpu_search_bool_packed(gix.handle, carr, ncl, qarr, nq, k, args.threshold, 0, None, ctypes.c_void_p(stream),
                                                    pg.local.data_ptr()))
        if world > 1:
            pg.gather()
            pg.merge_on_device(ctx, stream)
            host_rec.copy_(pg.merged, non_blocking=True)
        else:
            host_rec.copy_(pg.local, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t[0])
    e2e_qps = nq * args.steps / e2e_s
    e2e_gate = None
    if rank == 0 and not args.no_check:   # the e2e path returns the same page
        ed, es, ec, _, _ = unpack_record(host_rec.numpy(), nq, k)
        e2e_gate = gate(f"{args.workload} e2e N={world}", ed, es, ec, ref)["bit_exact"]

    extra = None
    if rank == 0 and world == 1 and not conj and not args.no_extra:
        extra = {"conj": conj_leg(args, searcher, sh, stream, max(5, args.steps // 2), threads, min(256, n_sample))}
    batch.close()
    gix.close()
    if rank == 0 and world == 1 and not conj and not args.no_extra:
        del sh
        ctx.close()
        ctx = None
        extra["knn"] = knn_leg(args, 0, 1, local_rank, max(5, args.steps // 4), 2)

    if rank == 0:
        pk, peak_src = peaks()
        peak = pk["hbm_gbs"]
        per_gpu_postings = alg_postings_total / world
        if conj:
            alg_bytes = per_gpu_postings * 8 + nq * k * 8   # + the intersection gathers, reported by the default line's extra.conj
        else:
            alg_bytes = per_gpu_postings * ALG_BYTES_PER_POSTING + nq * k * 8   # per launch (per GPU)
        traffic, traffic_src = (None, None)
        exh_traffic = None
        if world == 1 and not conj and args.docs == 10_000_000 and args.vocab == 1_000_000 and nq == 1024 and k == 100 and args.threshold == 1000:
            traffic, traffic_src = static_traffic("posting_probe_kernel<simple> TOP_SCORES")
            exh_traffic, _ = static_traffic("posting_probe_kernel<simple> COMPLETE")
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
        kernel_name = ("posting_probe_kernel<generic>" if conj else "posting_probe_kernel<simple>") + \
            " (persistent, data-parallel over the driver postings: 2-bit tf-plane gathers / granule-narrowed searches of TMA-staged lists, MAXSCORE roles, BM25 + exact top-k)"
        line = {
            "metric": "BM25 queries/sec (batch 1024, 10M docs)", "value": qps, "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, args.workload),
            "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "gate_bit_exact": e2e_gate},
            "gpu_launches": stats["launches_per_run"] * args.steps + (args.steps if world > 1 else 0),
            "gate": gate_info,
            "roofline": {"bound": "hbm", "kernel": kernel_name,
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "frac_kind": "effective: ALGORITHMIC bytes of every posting of the batch (9 B each, SURVEY.md 8d) / kernel time; MAXSCORE lets the kernel skip most of them, as the reference does",
                         "traffic": traffic, "traffic_source": traffic_src,
                         "physical_frac": None if traffic is None else traffic / (kernel_ms * 1e-3) / 1e9 / peak,
                         "peak_source": peak_src, "kernel_ms": kernel_ms, "merge_ms": merge_ms,
                         "alg_bytes_per_launch": alg_bytes, "alg_postings_per_launch": per_gpu_postings,
                         "mode": ("TOP_SCORES (totalHitsThreshold %d, the reference default)" % args.threshold) if args.threshold != INT_MAX else "COMPLETE (exact counts)",
                         "exhaustive": None if exh_ms is None else
                                       {"mode": "ScoreMode.COMPLETE: exact totalHits for every query (inclusion by ownership; a dense non-essential list contributes its posting count unread)",
                                        "kernel_ms": exh_ms, "achieved": alg_bytes / (exh_ms * 1e-3) / 1e9,
                                        "frac": alg_bytes / (exh_ms * 1e-3) / 1e9 / peak, "traffic": exh_traffic,
                                        "physical_frac": None if exh_traffic is None else exh_traffic / (exh_ms * 1e-3) / 1e9 / peak}},
            "cpu_baseline": cpu,
            "clocks": clocks,
            "index": {"postings": n_postings, "device_bytes": dev_bytes, "build_s": build_s, "work_items": stats["work_items"]},
            "extra": extra,
        }
        print(json.dumps(line))
        if outputs:
            dump_outputs(args.dump_outputs, outputs)
    if ctx is not None:
        ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
