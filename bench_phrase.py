"""Phrase-query benchmark, workload P1: prints one JSON line.

P1: a seeded corpus of --docs documents (2 000 000 by default) with lengths round(LogNormal(5.0, 0.8)) clipped to
[2, 20 000], tokens i.i.d. over a 1 000 000-term vocabulary with P(rank r) ~ 1/r, fieldnorm = length; postings
(WithFreqsAndPositions) and positions written by the library's writers.  Queries: --queries two-term and --queries
three-term phrases (PhraseQuery::new, slop 0), each the consecutive tokens at a uniformly drawn corpus position inside one
document, redrawn unless every rank lies in [10, 100 000], so every query matches; top k = 100.  The index is far larger
than the L2, so timed passes are not L2-resident.

Reported per batch: kernel ms (CUDA events inside the library: k_phrase_docs + k_phrase_match + k_and3_select) and
end-to-end ms (host clock around the call, which synchronises), medians over --steps after --warmup; queries/s; postings/s
(sum of the phrase terms' doc_freq / kernel time); the phrase terms' postings + positions bytes over kernel time as a fraction
of the HBM peak bench_bm25.py uses.  Parity: the first --check queries of each batch against a CPU restatement that reads the
raw token stream (not the positions file) on bench.host_threads() threads -- docs, order and f32 score bits equal, or exit 1.
Corpus generation time is reported separately."""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

VOCAB = 1_000_000


def gen_corpus(n_docs, seed):
    rng = np.random.default_rng(seed)
    lens = np.clip(np.rint(rng.lognormal(5.0, 0.8, n_docs)), 2, 20_000).astype(np.int64)
    cdf = np.cumsum(1.0 / np.arange(1, VOCAB + 1)); cdf /= cdf[-1]
    total = int(lens.sum())
    tok = np.empty(total, np.uint32)
    for a in range(0, total, 1 << 26):   # token = rank - 1
        b = min(total, a + (1 << 26))
        tok[a:b] = np.minimum(np.searchsorted(cdf, rng.random(b - a)), VOCAB - 1)
    return lens, tok


def build_index(lens, tok, threads):
    from stract_b200 import bm25
    n_docs = lens.size
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]])
    order = np.argsort(tok, kind="stable")                 # per term: ascending global position = (doc, position) order
    doc_of = np.repeat(np.arange(n_docs, dtype=np.uint32), lens)
    st = tok[order]; sd = doc_of[order]
    pos = (order - starts[sd]).astype(np.uint32)
    new = np.ones(order.size, bool); new[1:] = (st[1:] != st[:-1]) | (sd[1:] != sd[:-1])
    run_at = np.flatnonzero(new)
    docs = sd[run_at]; tfs = np.diff(np.append(run_at, order.size)).astype(np.uint32)
    term_off = np.searchsorted(st[run_at], np.arange(VOCAB + 1)).astype(np.uint64)
    fn_ids = bm25.fieldnorms_to_ids(lens)
    avg = np.float32(np.float32(int(lens.sum())) / np.float32(n_docs))
    post, infos = bm25.encode_postings_csr(docs, tfs, term_off, fn_ids, avg, threads=threads, record_option=2)
    pos_bytes, ps, pe = bm25.encode_positions_csr(docs, tfs, term_off, pos, threads=threads)
    seg = bm25.SegmentReader(post, infos, fn_ids, record_option=2, total_num_tokens=int(lens.sum()), positions=(pos_bytes, ps, pe))
    plen = np.array([infos[i].postings_len for i in range(VOCAB)], np.uint64)
    return seg, order, doc_of, plen, (pe - ps).astype(np.uint64)


def draw_phrases(rng, lens, tok, n, L):
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]]); ends = starts + lens
    out = []
    while len(out) < n:
        g = rng.integers(0, tok.size, 4 * n)
        d = np.searchsorted(ends, g, side="right")
        ok = g + L <= ends[d]
        for x in g[ok]:
            r = tok[x:x + L].astype(np.int64) + 1
            if r.min() >= 10 and r.max() <= 100_000:
                out.append([int(t) for t in tok[x:x + L]])
                if len(out) == n:
                    break
    return out


def oracle_phrase(terms, tok, order, tstart, doc_of, fn_ids, weight, cache, k):
    """slop-0 phrase counts straight from the token stream: starts g of terms[0] with tok[g + i] == terms[i] in the same doc."""
    g = order[tstart[terms[0]]:tstart[terms[0] + 1]]
    for i in range(1, len(terms)):
        g = g[g + i < tok.size]
        g = g[(tok[g + i] == terms[i]) & (doc_of[g + i] == doc_of[g])]
    d, c = np.unique(doc_of[g], return_counts=True)
    tf = c.astype(np.float32)
    sc = (np.float32(weight) * (tf / (tf + cache[fn_ids[d]]))).astype(np.float32)
    o = np.lexsort((d, -sc.astype(np.float64)))[:k]
    return d[o].astype(np.uint32), sc[o]


def gpu_name_power():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--docs", type=int, default=2_000_000)
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--check", type=int, default=2048)
    ap.add_argument("--seed", type=int, default=2024)
    a = ap.parse_args()
    import bench
    from stract_b200 import bm25
    threads = bench.host_threads()
    peaks, _ = bench._peaks()
    t0 = time.perf_counter()
    lens, tok = gen_corpus(a.docs, a.seed)
    seg, order, doc_of, plen, poslen = build_index(lens, tok, threads)
    gen_s = time.perf_counter() - t0
    tstart = np.searchsorted(tok[order], np.arange(VOCAB + 1))
    rng = np.random.default_rng(a.seed + 1)
    cache = bm25.compute_tf_cache(seg.average_fieldnorm)
    result = {"workload": "P1", "docs": a.docs, "tokens": int(tok.size), "k": a.k, "gen_s": round(gen_s, 1),
              "index_hbm_bytes": seg.info()["hbm_bytes"], "host_threads": threads}
    parity = True
    for L in (2, 3):
        phrases = draw_phrases(rng, lens, tok, a.queries, L)
        queries = [bm25.PhraseQuery(p) for p in phrases]
        weights = np.array([bm25.Bm25Weight.for_terms([int(seg.doc_freq[t]) for t in p], seg.max_doc, seg.average_fieldnorm).weight
                            for p in phrases], np.float32)
        td = bm25.TopDocs.with_limit(a.k)
        kern, e2e = [], []
        for step in range(a.warmup + a.steps):
            t1 = time.perf_counter()
            d, s, n, st = td.search_phrase_batch(seg, queries, weights=weights, return_stats=True)
            t2 = time.perf_counter()
            if step >= a.warmup:
                kern.append(st["kernel_ms"]); e2e.append((t2 - t1) * 1e3)
        km, em = float(np.median(kern)), float(np.median(e2e))
        alg = float(sum(int(plen[t]) + int(poslen[t]) for p in phrases for t in p))
        nchk = min(a.check, len(phrases))
        t3 = time.perf_counter()
        with ThreadPoolExecutor(threads) as ex:
            want = list(ex.map(lambda i: oracle_phrase(phrases[i], tok, order, tstart, doc_of, seg.fieldnorm_ids, weights[i], cache, a.k),
                               range(nchk)))
        cpu_s = time.perf_counter() - t3
        bad = 0
        for i, (wd, ws) in enumerate(want):
            if not (int(n[i]) == wd.size and np.array_equal(d[i, :n[i]], wd) and np.array_equal(s[i, :n[i]].view(np.uint32), ws.view(np.uint32))):
                bad += 1
        parity &= bad == 0
        result[f"phrase{L}"] = {"queries": len(phrases), "kernel_ms": km, "e2e_ms": em, "queries_per_s": len(phrases) / (em * 1e-3),
                                "postings_scored": st["postings_scored"], "postings_per_s": st["postings_scored"] / (km * 1e-3),
                                "candidates": st["docs_scored"], "alg_bytes": alg, "alg_gbs": alg / (km * 1e-3) / 1e9,
                                "hbm_frac": alg / (km * 1e-3) / 1e9 / peaks["hbm_gbs"], "hbm_peak_gbs": peaks["hbm_gbs"],
                                "matches": int(n.sum()), "cpu_oracle_queries": nchk, "cpu_oracle_s": round(cpu_s, 2),
                                "cpu_oracle_queries_per_s": nchk / cpu_s, "parity_mismatches": bad}
    name, power = gpu_name_power()
    result["gpu"] = name; result["power_limit"] = power; result["parity"] = "green" if parity else "red"
    print(json.dumps(result))
    seg.close()
    sys.exit(0 if parity else 1)


if __name__ == "__main__":
    main()
