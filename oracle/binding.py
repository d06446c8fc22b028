"""ctypes binding of oracle/liboracle.so (build: `make -C oracle`). TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None

i32p, i64p, f32p, u8p = (C.POINTER(t) for t in (C.c_int32, C.c_int64, C.c_float, C.c_uint8))


class OrcClause(C.Structure):
    _fields_ = [("occur", C.c_int32), ("kind", C.c_int32), ("id", C.c_int32), ("boost", C.c_float),
                ("lo", C.c_int64), ("hi", C.c_int64)]


class OrcQuery(C.Structure):
    _fields_ = [("clause_begin", C.c_int32), ("clause_end", C.c_int32), ("min_should_match", C.c_int32),
                ("has_after", C.c_int32), ("after_doc", C.c_int32), ("after_score", C.c_float)]


class OrcSort(C.Structure):
    _fields_ = [("kind", C.c_int32), ("column", C.c_int32), ("reverse", C.c_int32), ("reserved", C.c_int32),
                ("missing_value", C.c_int64)]


class OrcIndex(C.Structure):
    _fields_ = [
        ("n_docs", C.c_int32), ("doc_base", C.c_int32), ("n_terms", C.c_int32),
        ("term_off", i64p), ("post_docs", i32p), ("post_freqs", i32p), ("term_field", i32p), ("term_df", i64p),
        ("n_fields", C.c_int32), ("norms", C.POINTER(u8p)), ("field_doc_count", i64p), ("field_sum_ttf", i64p),
        ("field_k1", f32p), ("field_b", f32p),
        ("n_columns", C.c_int32), ("columns", C.POINTER(i64p)), ("column_has", C.POINTER(u8p)),
        ("live_docs", u8p), ("term_max_x", f32p), ("column_offsets", C.POINTER(i64p)),
    ]


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "liboracle.so")
    src = [os.path.join(_HERE, f) for f in ("oracle.c", "oracle.h", "Makefile")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


def _load_native():
    """liboracle.so rebuilt with -O3 -march=native for the host it runs on (bench.py's cpu_baseline / reference arm: the
    portable build that travels to the GPU box is -march=x86-64-v2). Same sources, same results (-ffp-contract=off, no
    fast-math). It is compiled in a temporary directory, so the source tree may be read-only; returns None (the caller
    keeps the portable build) when no compiler is present."""
    try:
        with tempfile.TemporaryDirectory(prefix="nrt_oracle_") as tmp:
            so = os.path.join(tmp, "liboracle_native.so")
            subprocess.check_call(["gcc", "-O3", "-march=native", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-fopenmp", "-std=c11",
                                   "-shared", "-o", so, os.path.join(_HERE, "oracle.c"), "-lm"], stderr=subprocess.DEVNULL)
            return C.CDLL(so)   # the loaded mapping outlives the file
    except Exception:
        return None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        so = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(so):
            build()
        L = (_load_native() if os.environ.get("NRT_ORACLE_NATIVE") == "1" else None) or C.CDLL(so)
        L.orc_int_to_byte4.restype = C.c_uint8
        L.orc_int_to_byte4.argtypes = [C.c_int32]
        L.orc_byte4_to_int.restype = C.c_int32
        L.orc_byte4_to_int.argtypes = [C.c_uint8]
        L.orc_bm25_idf.restype = C.c_float
        L.orc_bm25_idf.argtypes = [C.c_int64, C.c_int64]
        L.orc_bm25_avgdl.restype = C.c_float
        L.orc_bm25_avgdl.argtypes = [C.c_int64, C.c_int64]
        L.orc_bm25_cache.restype = None
        L.orc_bm25_cache.argtypes = [C.c_float, C.c_float, C.c_float, f32p]
        L.orc_bm25_score.restype = C.c_float
        L.orc_bm25_score.argtypes = [C.c_float, C.c_float, C.c_uint8, f32p]
        L.orc_build_term_max_x.restype = None
        L.orc_build_term_max_x.argtypes = [C.POINTER(OrcIndex), C.c_void_p]
        L.orc_search.argtypes = [C.POINTER(OrcIndex), C.POINTER(OrcClause), C.POINTER(OrcQuery), C.c_int32, C.c_int32,
                                 C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p]
        L.orc_search_limits.argtypes = [C.POINTER(OrcIndex), C.POINTER(OrcClause), C.POINTER(OrcQuery), C.c_int32, C.c_int32,
                                        C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_search_sorted.argtypes = [C.POINTER(OrcIndex), C.POINTER(OrcClause), C.POINTER(OrcQuery), C.c_int32, C.c_int32,
                                        C.c_int32, C.POINTER(OrcSort), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_match_bitmap.argtypes = [C.POINTER(OrcIndex), C.POINTER(OrcClause), C.POINTER(OrcQuery), C.c_void_p]
        L.orc_score_docs.argtypes = [C.POINTER(OrcIndex), C.POINTER(OrcClause), C.POINTER(OrcQuery), C.c_int32, C.c_int32, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_merge_topk.restype = None
        L.orc_merge_topk.argtypes = [C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 6
        L.orc_vector_score_f32.restype = C.c_float
        L.orc_vector_score_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
        L.orc_knn_exact.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_blend_rrf.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]
        L.orc_blend_scores.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                       C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]
        L.orc_rescore_combine.restype = None
        L.orc_rescore_combine.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_double, C.c_double]
        _lib = L
    return _lib


def int_to_byte4(i: int) -> int:
    return int(lib().orc_int_to_byte4(i))


def byte4_to_int(b: int) -> int:
    return int(lib().orc_byte4_to_int(b))


def bm25_idf(df: int, doc_count: int) -> np.float32:
    return np.float32(lib().orc_bm25_idf(df, doc_count))


def bm25_cache(k1: float, b: float, avgdl: float) -> np.ndarray:
    out = np.zeros(256, np.float32)
    lib().orc_bm25_cache(k1, b, avgdl, out.ctypes.data_as(f32p))
    return out


def bm25_term_score(boost: float, df: int, doc_count: int, sum_ttf: int, freq: int, length: int,
                    k1: float = 1.2, b: float = 0.75) -> np.float32:
    """Single-term score of a doc with `freq` occurrences and field length `length`."""
    L = lib()
    cache = bm25_cache(k1, b, float(L.orc_bm25_avgdl(sum_ttf, doc_count)))
    w = np.float32(np.float32(boost) * np.float32(L.orc_bm25_idf(df, doc_count)))
    return np.float32(L.orc_bm25_score(w, float(freq), int_to_byte4(length), cache.ctypes.data_as(f32p)))


class OracleIndex:
    """Wraps a nrtsearch_b200.index.HostShard-like object (duck-typed) for orc_search."""

    def __init__(self, sh, with_impacts: bool = False):
        self.keep = []

        def arr(a, dt):
            if a is None:
                return None
            b = np.ascontiguousarray(a, dtype=dt)
            self.keep.append(b)
            return b

        def ptr(a, typ):
            return C.cast(None, typ) if a is None else a.ctypes.data_as(typ)

        ix = OrcIndex()
        ix.n_docs, ix.doc_base, ix.n_terms = sh.n_docs, sh.doc_base, len(sh.term_off) - 1
        ix.term_off = ptr(arr(sh.term_off, np.int64), i64p)
        ix.post_docs = ptr(arr(sh.post_docs, np.int32), i32p)
        ix.post_freqs = ptr(arr(sh.post_freqs, np.int32), i32p)
        ix.term_field = ptr(arr(sh.term_field, np.int32), i32p)
        ix.term_df = ptr(arr(sh.term_df, np.int64), i64p)
        nf = len(sh.fields)
        ix.n_fields = nf
        norms = (u8p * max(nf, 1))()
        for i, f in enumerate(sh.fields):
            norms[i] = ptr(arr(f.norms, np.uint8), u8p)
        self.keep.append(norms)
        ix.norms = C.cast(norms, C.POINTER(u8p))
        ix.field_doc_count = ptr(arr(np.array([f.doc_count for f in sh.fields], np.int64), np.int64), i64p)
        ix.field_sum_ttf = ptr(arr(np.array([f.sum_total_term_freq for f in sh.fields], np.int64), np.int64), i64p)
        ix.field_k1 = ptr(arr(np.array([f.k1 for f in sh.fields], np.float32), np.float32), f32p)
        ix.field_b = ptr(arr(np.array([f.b for f in sh.fields], np.float32), np.float32), f32p)
        nc = len(sh.columns)
        ix.n_columns = nc
        cols = (i64p * max(nc, 1))()
        has = (u8p * max(nc, 1))()
        for i, c in enumerate(sh.columns):
            cols[i] = ptr(arr(c, np.int64), i64p)
            h = sh.column_has[i] if i < len(sh.column_has) else None
            has[i] = ptr(arr(h, np.uint8), u8p)
        offs = (i64p * max(nc, 1))()
        mv = getattr(sh, "column_offsets", None) or []
        for i in range(nc):
            o = mv[i] if i < len(mv) else None
            offs[i] = ptr(arr(o, np.int64), i64p)
        self.keep += [cols, has, offs]
        ix.columns = C.cast(cols, C.POINTER(i64p))
        ix.column_has = C.cast(has, C.POINTER(u8p))
        ix.column_offsets = C.cast(offs, C.POINTER(i64p))
        ix.live_docs = ptr(arr(sh.live_docs, np.uint8), u8p)
        ix.term_max_x = C.cast(None, f32p)
        self.ix = ix
        if with_impacts:
            mx = np.zeros(ix.n_terms, np.float32)
            lib().orc_build_term_max_x(C.byref(ix), mx.ctypes.data)
            self.keep.append(mx)
            ix.term_max_x = mx.ctypes.data_as(f32p)


def search(oix: OracleIndex, clauses, queries, top_k: int, total_hits_threshold: int = 2**31 - 1, mode: int = 0,
           n_threads: int = 0):
    """clauses: list of (occur, kind, id, boost, lo, hi); queries: list of (begin, end, msm, has_after, after_doc, after_score).
    Returns docs[nq,k], scores[nq,k], counts[nq], total[nq], relation[nq]."""
    nq = len(queries)
    carr = (OrcClause * max(len(clauses), 1))()
    for i, c in enumerate(clauses):
        carr[i] = OrcClause(*c)
    qarr = (OrcQuery * max(nq, 1))()
    for i, q in enumerate(queries):
        qarr[i] = OrcQuery(*q)
    docs = np.zeros((nq, top_k), np.int32)
    scores = np.zeros((nq, top_k), np.float32)
    counts = np.zeros(nq, np.int32)
    total = np.zeros(nq, np.int64)
    rel = np.zeros(nq, np.uint8)
    rc = lib().orc_search(C.byref(oix.ix), carr, qarr, nq, top_k, total_hits_threshold, mode, n_threads,
                          docs.ctypes.data, scores.ctypes.data, counts.ctypes.data, total.ctypes.data, rel.ctypes.data)
    if rc != 0:
        raise ValueError(f"orc_search failed ({rc})")
    return docs, scores, counts, total, rel


def search_compiled(oix: OracleIndex, carr, ncl: int, qarr, nq: int, top_k: int, total_hits_threshold: int = 2**31 - 1,
                    mode: int = 0, n_threads: int = 0):
    """Same, taking the ctypes arrays nrtsearch_b200.search.compile_queries produced (identical layouts)."""
    docs = np.zeros((nq, top_k), np.int32)
    scores = np.zeros((nq, top_k), np.float32)
    counts = np.zeros(nq, np.int32)
    total = np.zeros(nq, np.int64)
    rel = np.zeros(nq, np.uint8)
    rc = lib().orc_search(C.byref(oix.ix), C.cast(carr, C.POINTER(OrcClause)), C.cast(qarr, C.POINTER(OrcQuery)), nq,
                          top_k, total_hits_threshold, mode, n_threads, docs.ctypes.data, scores.ctypes.data,
                          counts.ctypes.data, total.ctypes.data, rel.ctypes.data)
    if rc != 0:
        raise ValueError(f"orc_search failed ({rc})")
    return docs, scores, counts, total, rel


def search_terminate_after(oix: OracleIndex, carr, ncl: int, qarr, nq: int, top_k: int, terminate_after: int,
                           max_recall: int = 0, n_threads: int = 0):
    """TerminateAfterWrapper semantics, sequential (doc order). Returns docs, scores, counts, total, relation, terminated."""
    docs = np.zeros((nq, top_k), np.int32)
    scores = np.zeros((nq, top_k), np.float32)
    counts = np.zeros(nq, np.int32)
    total = np.zeros(nq, np.int64)
    rel = np.zeros(nq, np.uint8)
    term = np.zeros(nq, np.uint8)
    rc = lib().orc_search_limits(C.byref(oix.ix), C.cast(carr, C.POINTER(OrcClause)), C.cast(qarr, C.POINTER(OrcQuery)), nq,
                                 top_k, 2**31 - 1, 0, n_threads, terminate_after, max_recall, docs.ctypes.data,
                                 scores.ctypes.data, counts.ctypes.data, total.ctypes.data, rel.ctypes.data, term.ctypes.data)
    if rc != 0:
        raise ValueError(f"orc_search_limits failed ({rc})")
    return docs, scores, counts, total, rel, term


def search_sorted(oix: OracleIndex, carr, ncl: int, qarr, nq: int, top_k: int, kind: int, column: int = 0, reverse: bool = False,
                  missing_value: int = 0, after_values=None, n_threads: int = 0):
    """TopFieldCollector semantics: returns docs [nq,k], sort values [nq,k] (int64), counts, total hits."""
    docs = np.zeros((nq, top_k), np.int32)
    vals = np.zeros((nq, top_k), np.int64)
    counts = np.zeros(nq, np.int32)
    total = np.zeros(nq, np.int64)
    st = OrcSort(kind, column, 1 if reverse else 0, 0, missing_value)
    av = None if after_values is None else np.ascontiguousarray(after_values, np.int64)
    rc = lib().orc_search_sorted(C.byref(oix.ix), C.cast(carr, C.POINTER(OrcClause)), C.cast(qarr, C.POINTER(OrcQuery)), nq, top_k,
                                 n_threads, C.byref(st), None if av is None else av.ctypes.data, docs.ctypes.data, vals.ctypes.data,
                                 counts.ctypes.data, total.ctypes.data)
    if rc != 0:
        raise ValueError(f"orc_search_sorted failed ({rc})")
    return docs, vals, counts, total


def match_bitmap(oix: OracleIndex, carr, qarr, qi: int) -> np.ndarray:
    """0/1 per doc: the docs query qi matches (the stream the reference's additional collectors see)."""
    out = np.zeros(oix.ix.n_docs, np.uint8)
    q = C.cast(qarr, C.POINTER(OrcQuery))
    rc = lib().orc_match_bitmap(C.byref(oix.ix), C.cast(carr, C.POINTER(OrcClause)), C.byref(q[qi]), out.ctypes.data)
    if rc != 0:
        raise ValueError("orc_match_bitmap failed")
    return out


def score_docs(oix: OracleIndex, carr, qarr, nq: int, docs, counts=None):
    docs = np.ascontiguousarray(docs, np.int32)
    n_hits = docs.shape[1]
    cn = None if counts is None else np.ascontiguousarray(counts, np.int32)
    m = np.zeros((nq, n_hits), np.uint8)
    s = np.zeros((nq, n_hits), np.float32)
    rc = lib().orc_score_docs(C.byref(oix.ix), C.cast(carr, C.POINTER(OrcClause)), C.cast(qarr, C.POINTER(OrcQuery)), nq, n_hits,
                              docs.ctypes.data, None if cn is None else cn.ctypes.data, m.ctypes.data, s.ctypes.data)
    if rc != 0:
        raise ValueError("orc_score_docs failed")
    return m, s


def merge_topk(docs, scores, counts, top_k):
    """docs/scores [n_lists, nq, top_k], counts [n_lists, nq] -> merged docs, scores, counts."""
    docs = np.ascontiguousarray(docs, np.int32)
    scores = np.ascontiguousarray(scores, np.float32)
    counts = np.ascontiguousarray(counts, np.int32)
    nl, nq, _ = docs.shape
    od, os_, oc = np.zeros((nq, top_k), np.int32), np.zeros((nq, top_k), np.float32), np.zeros(nq, np.int32)
    lib().orc_merge_topk(nl, nq, top_k, docs.ctypes.data, scores.ctypes.data, counts.ctypes.data, od.ctypes.data,
                         os_.ctypes.data, oc.ctypes.data)
    return od, os_, oc


def vector_score(a, b, sim: int) -> np.float32:
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    return np.float32(lib().orc_vector_score_f32(a.ctypes.data, b.ctypes.data, len(a), sim))


def knn_exact(corpus, sim: int, queries, k: int, doc_base: int = 0, filter_docs=None, boosts=None, n_threads: int = 0,
              live_docs=None):
    corpus = np.ascontiguousarray(corpus, np.float32)
    queries = np.ascontiguousarray(queries, np.float32)
    n, dims = corpus.shape
    nq = queries.shape[0]
    f = None if filter_docs is None else np.ascontiguousarray(filter_docs, np.uint8)
    b = None if boosts is None else np.ascontiguousarray(boosts, np.float32)
    lv = None if live_docs is None else np.ascontiguousarray(live_docs, np.uint8)
    docs, scores, counts = np.zeros((nq, k), np.int32), np.zeros((nq, k), np.float32), np.zeros(nq, np.int32)
    rc = lib().orc_knn_exact(corpus.ctypes.data, n, dims, sim, doc_base, None if f is None else f.ctypes.data,
                             queries.ctypes.data, nq, None if b is None else b.ctypes.data, k, n_threads,
                             docs.ctypes.data, scores.ctypes.data, counts.ctypes.data, None if lv is None else lv.ctypes.data)
    if rc != 0:
        raise ValueError("orc_knn_exact failed")
    return docs, scores, counts


def blend_rrf(docs, counts, boosts, rank_constant: int, top_out: int):
    docs = np.ascontiguousarray(docs, np.int32)
    counts = np.ascontiguousarray(counts, np.int32)
    boosts = np.ascontiguousarray(boosts, np.float32)
    R, top_in = docs.shape
    od, os_ = np.zeros(top_out, np.int32), np.zeros(top_out, np.float32)
    total = C.c_int32()
    n = lib().orc_blend_rrf(R, top_in, docs.ctypes.data, counts.ctypes.data, boosts.ctypes.data, rank_constant, top_out,
                            od.ctypes.data, os_.ctypes.data, C.byref(total))
    return od[:n], os_[:n], total.value


def blend_scores(mode: int, docs, scores, counts, boosts, top_out: int):
    """Score-order blend of one query: docs/scores [R, top_in], mode 1 MAX / 2 SUM / 3 AVG."""
    docs = np.ascontiguousarray(docs, np.int32)
    scores = np.ascontiguousarray(scores, np.float32)
    counts = np.ascontiguousarray(counts, np.int32)
    boosts = np.ascontiguousarray(boosts, np.float32)
    R, top_in = docs.shape
    od, os_ = np.zeros(top_out, np.int32), np.zeros(top_out, np.float32)
    total = C.c_int32()
    n = lib().orc_blend_scores(mode, R, top_in, docs.ctypes.data, scores.ctypes.data, counts.ctypes.data, boosts.ctypes.data, top_out,
                               od.ctypes.data, os_.ctypes.data, C.byref(total))
    return od[:n], os_[:n], total.value


def rescore_combine(docs, scores, second_matches, second_scores, query_weight: float, rescore_weight: float):
    docs = np.ascontiguousarray(docs, np.int32).copy()
    scores = np.ascontiguousarray(scores, np.float32).copy()
    m = np.ascontiguousarray(second_matches, np.uint8)
    s2 = np.ascontiguousarray(second_scores, np.float32)
    lib().orc_rescore_combine(len(docs), len(docs), docs.ctypes.data, scores.ctypes.data, m.ctypes.data, s2.ctypes.data,
                              query_weight, rescore_weight)
    return docs, scores
