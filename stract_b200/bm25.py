"""Host-side mirror of the reference's BM25 top-k interface, backed by libstract_b200.so.

Mirrors (same names / argument meaning):
  fieldnorm_to_id / id_to_fieldnorm       tantivy/src/fieldnorm/code.rs:1-11
  Bm25Weight.for_one_term / for_terms / idf  tantivy/src/query/bm25.rs:52-176   (f32 arithmetic, host side)
  StractBm25Weight                          core/src/ranking/bm25.rs:23-151
  PostingsWriter                            tantivy/src/postings/serializer.rs (WithFreqs) -- builds segments
  SegmentReader.open                        InvertedIndexReader + FieldNormReader of one field
  TopDocs.with_limit(k) + BooleanQuery      tantivy/src/collector/top_score_collector.rs:360-414
  PhraseQuery (slop 0) + TopDocs            tantivy/src/query/phrase_query/*.rs, positions/*.rs
  SignalComputer (one text field + numeric signals)   core/src/ranking/computer/mod.rs, initial.rs:79-93

The weights are computed on the host exactly like the reference does before it opens any posting list
(f32 `ln` once per term); all per-posting work runs in the CUDA library.
"""
import ctypes as C
import math

import numpy as np

from . import _lib_bm25 as B
from ._lib import check, lib
from ._hostmem import host_out

K1 = np.float32(1.2)
B_ = np.float32(0.75)
MODE_AND, MODE_OR, MODE_OR_WAND = 0, 1, 2   # MODE_OR_WAND: block_wand replayed, bit-exact sums for >= 3 terms
NO_TERM = 0xFFFFFFFF


def id_to_fieldnorm(i):
    return int(lib().sb200_fieldnorm_id_to_value(int(i)))


def fieldnorm_to_id(v):
    return int(lib().sb200_fieldnorm_value_to_id(int(v)))


_TABLE = None


def fieldnorm_table():
    global _TABLE
    if _TABLE is None:
        _TABLE = np.array([id_to_fieldnorm(i) for i in range(256)], np.uint32)
    return _TABLE


def fieldnorms_to_ids(fieldnorms):
    return (np.searchsorted(fieldnorm_table(), np.asarray(fieldnorms, np.uint32), side="right") - 1).astype(np.uint8)


def idf(doc_freq, doc_count):
    """tantivy/src/query/bm25.rs:52-56 in f32 (f32 `ln` through libm, like Rust's f32::ln)."""
    assert doc_count >= doc_freq
    x = (np.float32(doc_count - doc_freq) + np.float32(0.5)) / (np.float32(doc_freq) + np.float32(0.5))
    return np.float32(_logf(np.float32(1.0) + x))


_libm = C.CDLL("libm.so.6")
_libm.logf.restype = C.c_float
_libm.logf.argtypes = [C.c_float]


def _logf(x):
    return _libm.logf(float(x))


def idf_array(doc_freq, doc_count, tantivy_weight=False):
    """idf (or Bm25Weight.weight = idf * (1 + K1)) for an array of doc_freqs through the library's host helper: the same f32
    expression and C-library logf as `idf`, without an interpreter round trip per value."""
    df = np.ascontiguousarray(doc_freq, np.uint32)
    out = np.empty(df.shape, np.float32)
    check(lib().sb200_bm25_idf(df.ctypes.data, df.size, int(doc_count), 1 if tantivy_weight else 0, out.ctypes.data))
    return out


def compute_tf_cache(average_fieldnorm, k1=K1, b=B_):
    """cache[id] = K1 * (1 - B + B * fieldnorm(id) / avg) (bm25.rs:58-68), f32 left to right."""
    fn = fieldnorm_table().astype(np.float32)
    avg = np.float32(average_fieldnorm)
    k1 = np.float32(k1); b = np.float32(b)
    return (k1 * ((np.float32(1.0) - b) + (b * fn) / avg)).astype(np.float32)


class Bm25Weight:
    """tantivy Bm25Weight: weight = idf * (1 + K1), score = weight * (tf / (tf + cache[fieldnorm_id]))."""

    def __init__(self, idf_value, average_fieldnorm):
        self.weight = np.float32(np.float32(idf_value) * (np.float32(1.0) + K1))
        self.cache = compute_tf_cache(average_fieldnorm)
        self.average_fieldnorm = np.float32(average_fieldnorm)

    @classmethod
    def for_one_term(cls, term_doc_freq, total_num_docs, avg_fieldnorm):
        return cls(idf(term_doc_freq, total_num_docs), avg_fieldnorm)

    @classmethod
    def for_terms(cls, doc_freqs, total_num_docs, avg_fieldnorm):
        """Bm25Weight::for_terms (bm25.rs:98-134): one term -> for_one_term; several -> the f32 sum of their idfs in the order
        given (a phrase's terms in offset order), so for three or more terms the order changes the bits."""
        doc_freqs = [int(d) for d in doc_freqs]
        if len(doc_freqs) == 1:
            return cls.for_one_term(doc_freqs[0], total_num_docs, avg_fieldnorm)
        acc = np.float32(0.0)
        for d in doc_freqs:
            acc = np.float32(acc + idf(d, total_num_docs))
        return cls(acc, avg_fieldnorm)

    def score(self, fieldnorm_id, term_freq):
        tf = np.float32(term_freq)
        return np.float32(self.weight * (tf / (tf + self.cache[fieldnorm_id])))


class StractBm25Weight:
    """core/src/ranking/bm25.rs:110-151: weight = idf, score = idf * ((tf*(k1+1)) / (tf + cache)), tf==0 -> 0."""

    def __init__(self, idf_value, average_fieldnorm, k1=K1, b=B_):
        self.weight = np.float32(idf_value)
        self.k1 = np.float32(k1)
        self.cache = compute_tf_cache(average_fieldnorm, k1, b)

    @classmethod
    def for_one_term(cls, term_doc_freq, total_num_docs, avg_fieldnorm, k1=K1, b=B_):
        return cls(idf(term_doc_freq, total_num_docs), avg_fieldnorm, k1, b)


def _p(a):
    return a.ctypes.data if a is not None else None


def encode_postings(term_docs, term_tfs, fieldnorm_ids, avg_fieldnorm, threads=8, record_option=1):
    """PostingsSerializer for a list of terms (record_option 1 = WithFreqs, 2 = WithFreqsAndPositions).  Returns
    (bytes u8[], TermInfo array)."""
    n = len(term_docs)
    off = np.zeros(n + 1, np.uint64)
    for i, d in enumerate(term_docs):
        off[i + 1] = off[i] + len(d)
    docs = np.concatenate([np.asarray(d, np.uint32) for d in term_docs]) if n else np.zeros(0, np.uint32)
    tfs = np.concatenate([np.asarray(t, np.uint32) for t in term_tfs]) if n else np.zeros(0, np.uint32)
    return encode_postings_csr(docs, tfs, off, fieldnorm_ids, avg_fieldnorm, threads, record_option)


def encode_postings_csr(docs, tfs, off, fieldnorm_ids, avg_fieldnorm, threads=8, record_option=1):
    L = lib()
    docs = np.ascontiguousarray(docs, np.uint32); tfs = np.ascontiguousarray(tfs, np.uint32)
    off = np.ascontiguousarray(off, np.uint64)
    fn = np.ascontiguousarray(fieldnorm_ids, np.uint8)
    n = off.size - 1
    ln = C.c_uint64(0)
    infos = (B.TermInfo * max(n, 1))()
    check(L.sb200_postings_encode_ex(_p(docs), _p(tfs), _p(off), n, _p(fn), fn.size, float(avg_fieldnorm), int(record_option),
                                     None, 0, C.byref(ln), None, threads))
    out = np.zeros(max(ln.value, 1), np.uint8)
    check(L.sb200_postings_encode_ex(_p(docs), _p(tfs), _p(off), n, _p(fn), fn.size, float(avg_fieldnorm), int(record_option),
                                     _p(out), out.size, C.byref(ln), infos, threads))
    return out[:ln.value], infos


def encode_positions(term_docs, term_tfs, term_positions, threads=8):
    """PositionSerializer for a list of terms: term_positions[t] holds the absolute positions of every posting of term t,
    posting after posting (sum(tfs) entries).  Returns (bytes u8[], pos_start u64[], pos_end u64[])."""
    n = len(term_docs)
    off = np.zeros(n + 1, np.uint64)
    for i, d in enumerate(term_docs):
        off[i + 1] = off[i] + len(d)
    cat = lambda xs: np.concatenate([np.asarray(x, np.uint32) for x in xs]) if n else np.zeros(0, np.uint32)  # noqa: E731
    return encode_positions_csr(cat(term_docs), cat(term_tfs), off, cat(term_positions), threads)


def encode_positions_csr(docs, tfs, off, positions, threads=8):
    L = lib()
    docs = np.ascontiguousarray(docs, np.uint32); tfs = np.ascontiguousarray(tfs, np.uint32)
    off = np.ascontiguousarray(off, np.uint64); positions = np.ascontiguousarray(positions, np.uint32)
    n = off.size - 1
    ln = C.c_uint64(0)
    check(L.sb200_positions_encode(_p(docs), _p(tfs), _p(off), n, _p(positions), None, 0, C.byref(ln), None, None, threads))
    out = np.zeros(max(ln.value, 1), np.uint8)
    ps = np.zeros(max(n, 1), np.uint64); pe = np.zeros(max(n, 1), np.uint64)
    check(L.sb200_positions_encode(_p(docs), _p(tfs), _p(off), n, _p(positions), _p(out), out.size, C.byref(ln), _p(ps), _p(pe), threads))
    return out[:ln.value], ps[:n], pe[:n]


def decode_term_info_store(store, device=0, with_positions=False):
    """TermInfoStore bytes (the `.term` store behind tantivy's FST term dictionary) -> TermInfo array, decoded on the
    device (sb200_term_info_store_decode); pass the result to SegmentReader.  with_positions=True also returns every
    term's positions range (pos_start, pos_end), what SegmentReader's `positions` takes."""
    L = lib()
    store = np.ascontiguousarray(store, np.uint8)
    n = C.c_uint64(0)
    check(L.sb200_term_info_store_decode(_p(store), store.size, device, None, 0, C.byref(n)))
    infos = (B.TermInfo * max(n.value, 1))()
    check(L.sb200_term_info_store_decode(_p(store), store.size, device, infos, n.value, C.byref(n)))
    if not with_positions:
        return infos, int(n.value)
    ps = np.zeros(max(n.value, 1), np.uint64); pe = np.zeros(max(n.value, 1), np.uint64)
    check(L.sb200_term_info_store_decode_positions(_p(store), store.size, device, _p(ps), _p(pe), n.value, C.byref(n)))
    return infos, int(n.value), (ps[:n.value], pe[:n.value])


class SegmentReader:
    """One field of one segment resident in HBM (postings file + fieldnorms + block directory)."""

    def __init__(self, postings, term_infos, fieldnorm_ids, device=0, record_option=1, total_num_tokens=None, positions=None):
        self._L = lib()
        self._h = C.c_void_p()
        postings = np.ascontiguousarray(postings, np.uint8)
        self.fieldnorm_ids = np.ascontiguousarray(fieldnorm_ids, np.uint8)
        self.max_doc = int(self.fieldnorm_ids.size)
        if isinstance(term_infos, tuple):  # (off, len, df) arrays
            o, l, d = term_infos
            arr = (B.TermInfo * max(len(d), 1))()
            for i in range(len(d)):
                arr[i].postings_off, arr[i].postings_len, arr[i].doc_freq = int(o[i]), int(l[i]), int(d[i])
            term_infos, n_terms = arr, len(d)
        else:
            n_terms = len(term_infos)
        self.n_terms = n_terms
        self.doc_freq = np.array([term_infos[i].doc_freq for i in range(n_terms)], np.uint32)
        check(self._L.sb200_segment_create(_p(postings), postings.size, term_infos, n_terms, _p(self.fieldnorm_ids), self.max_doc,
                                           record_option, device, C.byref(self._h)))
        if total_num_tokens is None:
            # tantivy keeps the exact token count in the inverted index (InvertedIndexReader::total_num_tokens); a caller that
            # opens a real segment must pass it.  The reconstruction from the quantised fieldnorm ids below is exact only for
            # indexes written from those ids (the synthetic / test segments of this repo).
            import warnings
            if not getattr(SegmentReader, "_warned_tokens", False):
                warnings.warn("SegmentReader: total_num_tokens not given; reconstructing it from the fieldnorm ids (exact only for "
                              "segments written from those ids)", stacklevel=2)
                SegmentReader._warned_tokens = True
            total_num_tokens = int(fieldnorm_table()[self.fieldnorm_ids].astype(np.uint64).sum())
        self.total_num_tokens = total_num_tokens
        # average_fieldnorm = total_num_tokens as f32 / total_num_docs as f32 (bm25.rs:112-114)
        self.average_fieldnorm = np.float32(np.float32(total_num_tokens) / np.float32(max(self.max_doc, 1)))
        self.device = device
        if positions is not None:
            self.attach_positions(*positions)

    def attach_positions(self, data, pos_start, pos_end):
        """The field's positions file and every term's byte range in it (sb200_segment_attach_positions); needs
        record_option=2 (WithFreqsAndPositions)."""
        data = np.ascontiguousarray(data, np.uint8)
        ps = np.ascontiguousarray(pos_start, np.uint64); pe = np.ascontiguousarray(pos_end, np.uint64)
        if ps.size != self.n_terms or pe.size != self.n_terms:
            raise ValueError(f"{self.n_terms} terms, {ps.size} / {pe.size} positions ranges")
        check(self._L.sb200_segment_attach_positions(self._h, _p(data), data.size, _p(ps), _p(pe)))

    def info(self):
        si = B.SegmentInfo()
        check(self._L.sb200_segment_get_info(self._h, C.byref(si)))
        return {k: getattr(si, k) for k, _ in B.SegmentInfo._fields_ if not k.startswith("_")}

    def close(self):
        if self._h:
            self._L.sb200_segment_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SignalTable:
    """Numeric signal scores per doc, row-major in HBM (sb200_signals)."""

    def __init__(self, columns, device=0):
        self._L = lib()
        self._h = C.c_void_p()
        cols = [np.ascontiguousarray(c, np.float64) for c in columns]
        self.n_cols = len(cols)
        self.max_doc = int(cols[0].size) if cols else 0
        arr = (C.c_void_p * max(self.n_cols, 1))(*[c.ctypes.data for c in cols])
        check(self._L.sb200_signals_create(arr, self.n_cols, self.max_doc, device, C.byref(self._h)))

    def close(self):
        if self._h:
            self._L.sb200_signals_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# The numeric signals of CoreSignalEnum in declaration order (core/src/ranking/signals/mod.rs:206-218) with the transform
# their `compute` applies to the fast-field value (core/src/ranking/signals/core/non_text.rs), the element type of the column
# and the default coefficient.
NUM_IDENTITY, NUM_RANK, NUM_BOOL, NUM_BOOL_NOT, NUM_INVERSE, NUM_FETCH_TIME, NUM_UPDATE_TIME, NUM_LINK_DENSITY, NUM_REGION = range(9)
NUM_U64, NUM_F64, NUM_BOOL8 = 0, 1, 2
NUMERIC_SIGNALS = [
    # name,               transform,        dtype,     default coefficient
    ("HostCentrality",     NUM_IDENTITY,     NUM_F64,   2.0),
    ("HostCentralityRank", NUM_RANK,         NUM_U64,   0.02),
    ("PageCentrality",     NUM_IDENTITY,     NUM_F64,   2.0),
    ("PageCentralityRank", NUM_RANK,         NUM_U64,   0.02),
    ("IsHomepage",         NUM_BOOL,         NUM_BOOL8, 0.01),
    ("FetchTimeMs",        NUM_FETCH_TIME,   NUM_U64,   0.001),
    ("UpdateTimestamp",    NUM_UPDATE_TIME,  NUM_U64,   0.75),
    ("TrackerScore",       NUM_INVERSE,      NUM_U64,   0.1),
    ("Region",             NUM_REGION,       NUM_U64,   0.15),
    ("UrlDigits",          NUM_INVERSE,      NUM_U64,   0.01),
    ("UrlSlashes",         NUM_INVERSE,      NUM_U64,   0.1),
    ("LinkDensity",        NUM_LINK_DENSITY, NUM_F64,   0.0),
    ("HasAds",             NUM_BOOL_NOT,     NUM_BOOL8, 0.01),
]


class RawSignalTable(SignalTable):
    """The numeric-signal score table built by the library from the RAW fast-field columns (sb200_signals_create_raw).

    `columns` = {signal name: raw column} (u64 / f64 / bool arrays as in NUMERIC_SIGNALS); the table's column order is
    CoreSignalEnum order.  `current_timestamp` feeds UpdateTimestamp (SignalComputer::set_current_timestamp), `region_count`
    = (counts per region id, total) feeds Region (RegionCount::score), `selected_region` the query's region boost.
    `numeric` is the [(name, column, default coefficient)] list SignalComputeOrder / MultiFieldSignalComputer take."""

    def __init__(self, columns, current_timestamp=None, region_count=None, selected_region=None, device=0):
        self._L = lib()
        self._h = C.c_void_p()
        names = [n for n, _, _, _ in NUMERIC_SIGNALS if n in columns]
        unknown = set(columns) - set(names)
        if unknown:
            raise KeyError(f"not numeric CoreSignals: {sorted(unknown)}")
        np_dt = {NUM_U64: np.uint64, NUM_F64: np.float64, NUM_BOOL8: np.uint8}
        arr = (B.NumericColumn * max(len(names), 1))()
        keep, self.numeric = [], []
        lut = None
        if region_count is not None:
            counts, total = region_count
            lut = np.array([0.0 if c is None else float(c) / float(total) for c in counts], np.float64)   # count as f64 / total as f64
        for i, n in enumerate(names):
            _, kind, dt, coef = next(e for e in NUMERIC_SIGNALS if e[0] == n)
            raw = np.ascontiguousarray(columns[n], np_dt[dt])
            keep.append(raw)
            arr[i].kind, arr[i].dtype, arr[i].raw = kind, dt, raw.ctypes.data
            if kind == NUM_UPDATE_TIME:
                arr[i].p0 = float(current_timestamp or 0)
            if kind == NUM_REGION and lut is not None:
                arr[i].lut, arr[i].lut_len = lut.ctypes.data, lut.size
                if selected_region is not None:
                    arr[i].p0, arr[i].p1 = float(selected_region), 1.0
            self.numeric.append((n, i, coef))
        self.n_cols = len(names)
        self.max_doc = int(keep[0].size) if keep else 0
        assert all(k.size == self.max_doc for k in keep)
        check(self._L.sb200_signals_create_raw(arr, self.n_cols, self.max_doc, device, C.byref(self._h)))

    def read(self, first_doc=0, n_docs=None):
        n = self.max_doc - first_doc if n_docs is None else n_docs
        out = np.zeros((n, self.n_cols), np.float64)
        check(self._L.sb200_signals_read(self._h, first_doc, n, out.ctypes.data))
        return out


def score_rank(rank):
    """non_text.rs:50-59: (10 - log_8(1 + rank)).max(0) with f64::log(base) = ln(x)/ln(base)."""
    return max(10.0 - math.log(1.0 + float(rank)) / math.log(8.0), 0.0)


class TopDocs:
    """`TopDocs::with_limit(k)` over a BooleanQuery of TermQueries on one field, batched."""

    def __init__(self, limit, offset=0):
        assert limit >= 1, "Limit must be strictly greater than 0."  # top_collector.rs:85
        self.limit = limit
        self.offset = offset

    @classmethod
    def with_limit(cls, limit):
        return cls(limit)

    def and_offset(self, offset):
        """TopDocs::and_offset (top_score_collector.rs:170-172): the segment collects limit + offset documents and the
        merged fruit drops the first `offset` (top_collector.rs:109-129)."""
        return TopDocs(self.limit, int(offset))

    def search_batch(self, segment, term_ords, mode=MODE_AND, weights=None, return_stats=False, average_fieldnorm=None):
        """term_ords [n_queries, n_terms] (NO_TERM pads).  Returns (docs [nq,k], scores [nq,k], n_out [nq]).
        `weights` / `average_fieldnorm` override the segment's own statistics (a Searcher passes the index-wide ones)."""
        term_ords = np.ascontiguousarray(term_ords, np.uint32)
        nq, nt = term_ords.shape
        if weights is None:  # Bm25Weight::for_terms with the segment's own statistics (bm25.rs:98-134)
            weights = idf_array(segment.doc_freq[np.minimum(term_ords, segment.n_terms - 1)], segment.max_doc, tantivy_weight=True)
        weights = np.ascontiguousarray(weights, np.float32)
        cache = compute_tf_cache(segment.average_fieldnorm if average_fieldnorm is None else average_fieldnorm)
        k = self.limit + self.offset
        docs = host_out((nq, k), np.uint32); scores = host_out((nq, k), np.float32); n_out = np.zeros(nq, np.uint32)
        b = B.Bm25Batch(nq, nt, _p(term_ords), _p(weights), _p(cache), mode, k)
        st = B.Bm25Stats()
        check(segment._L.sb200_bm25_topk_batch(segment._h, C.byref(b), _p(docs), _p(scores), _p(n_out), C.byref(st)))
        if self.offset:
            o = self.offset
            docs = np.ascontiguousarray(docs[:, o:]); scores = np.ascontiguousarray(scores[:, o:])
            n_out = (np.maximum(n_out.astype(np.int64) - o, 0)).astype(np.uint32)
        if return_stats:
            return docs, scores, n_out, {k_: getattr(st, k_) for k_, _ in B.Bm25Stats._fields_ if not k_.startswith("_")}
        return docs, scores, n_out

    def search_phrase_batch(self, segment, queries, weights=None, average_fieldnorm=None, return_stats=False):
        """A list of PhraseQuery on one segment (sb200_phrase_topk_batch).  Returns (docs [nq,k], scores [nq,k], n_out [nq]).
        `weights` ([nq] Bm25Weight.for_terms(..).weight) / `average_fieldnorm` override the segment's own statistics."""
        nq = len(queries)
        ords, offs, lens = _phrase_arrays(queries)
        if weights is None:
            weights = [Bm25Weight.for_terms([int(segment.doc_freq[t]) if t != NO_TERM else 0 for t in p.term_ords], segment.max_doc,
                                            segment.average_fieldnorm).weight for p in queries]
        w = np.zeros(max(nq, 1), np.float32); w[:nq] = np.asarray(weights, np.float32)
        cache = compute_tf_cache(segment.average_fieldnorm if average_fieldnorm is None else average_fieldnorm)
        k = self.limit + self.offset
        docs = host_out((max(nq, 1), k), np.uint32); scores = host_out((max(nq, 1), k), np.float32); n_out = np.zeros(max(nq, 1), np.uint32)
        b = B.PhraseBatch(nq, ords.shape[1], _p(ords), _p(offs), _p(lens), _p(w), _p(cache), k)
        st = B.Bm25Stats()
        check(segment._L.sb200_phrase_topk_batch(segment._h, C.byref(b), _p(docs), _p(scores), _p(n_out), C.byref(st)))
        docs, scores, n_out = docs[:nq], scores[:nq], n_out[:nq]
        if self.offset:
            o = self.offset
            docs = np.ascontiguousarray(docs[:, o:]); scores = np.ascontiguousarray(scores[:, o:])
            n_out = (np.maximum(n_out.astype(np.int64) - o, 0)).astype(np.uint32)
        if return_stats:
            return docs, scores, n_out, {k_: getattr(st, k_) for k_, _ in B.Bm25Stats._fields_ if not k_.startswith("_")}
        return docs, scores, n_out

    def search(self, segment, term_ords, mode=MODE_AND, weights=None):
        """One query -> list of (score, doc) like the Fruit Vec<(Score, DocAddress)>."""
        t = np.asarray(term_ords, np.uint32)[None, :]
        w = None if weights is None else np.asarray(weights, np.float32)[None, :]
        d, s, n = self.search_batch(segment, t, mode, w)
        return [(float(s[0, i]), int(d[0, i])) for i in range(int(n[0]))]


class PhraseQuery:
    """PhraseQuery::new(terms) / new_with_offset(terms_with_offset) (phrase_query.rs:35-53) with slop 0, terms as ordinals of
    one field (NO_TERM: absent from the segment).  The terms are kept sorted by offset (stable), as the reference keeps them."""

    def __init__(self, term_ords, offsets=None):
        term_ords = [int(t) for t in term_ords]
        offsets = list(range(len(term_ords))) if offsets is None else [int(o) for o in offsets]
        if len(term_ords) < 2:
            raise ValueError("A phrase query is required to have strictly more than one term.")
        if len(offsets) != len(term_ords):
            raise ValueError("one offset per term")
        pairs = sorted(zip(offsets, term_ords), key=lambda p: p[0])
        self.offsets = [o for o, _ in pairs]
        self.term_ords = [t for _, t in pairs]


def _phrase_arrays(queries):
    nq = len(queries)
    nt = max([2] + [len(p.term_ords) for p in queries])
    ords = np.full((max(nq, 1), nt), NO_TERM, np.uint32); offs = np.zeros((max(nq, 1), nt), np.uint32)
    lens = np.zeros(max(nq, 1), np.uint8)
    for q, p in enumerate(queries):
        ords[q, :len(p.term_ords)] = p.term_ords; offs[q, :len(p.offsets)] = p.offsets; lens[q] = len(p.term_ords)
    return ords, offs, lens


class Searcher:
    """tantivy `Searcher` + `TopDocs` over several segments of one field.  The BM25 statistics are the index-wide ones
    (Bm25StatisticsProvider / Bm25Weight::for_terms, tantivy/src/query/bm25.rs:15-50,98-134: total_num_docs,
    total_num_tokens and doc_freq summed over the segments); every segment collects limit + offset documents on the
    device and the fruits are merged by (score desc, DocAddress(segment_ord, doc_id) asc), then the offset is dropped
    (TopCollector::merge_fruits, tantivy/src/collector/top_collector.rs:109-129)."""

    def __init__(self, segments):
        self.segments = list(segments)
        self.total_num_docs = int(sum(s.max_doc for s in self.segments))
        self.total_num_tokens = int(sum(s.total_num_tokens for s in self.segments))
        self.average_fieldnorm = np.float32(np.float32(self.total_num_tokens) / np.float32(max(self.total_num_docs, 1)))

    def doc_freq(self, term_ords_per_segment):
        df = np.zeros(np.asarray(term_ords_per_segment[0]).shape, np.int64)
        for seg, ords in zip(self.segments, term_ords_per_segment):
            ords = np.asarray(ords, np.uint32)
            present = ords != NO_TERM
            df += np.where(present, seg.doc_freq[np.minimum(ords, max(seg.n_terms - 1, 0))].astype(np.int64), 0)
        return df

    def search_batch(self, top_docs, term_ords_per_segment, mode=MODE_AND, n_clauses=None):
        """term_ords_per_segment[s] is [n_queries, n_terms] in segment s's own ordinals, NO_TERM where the segment does not
        hold the term; n_clauses[q] = number of leading columns that are real clauses (default: all).  Returns
        (segment_ord [nq,k], docs [nq,k], scores [nq,k], n [nq])."""
        ords = [np.ascontiguousarray(o, np.uint32) for o in term_ords_per_segment]
        nq, nt = ords[0].shape
        n_clauses = np.full(nq, nt, np.int64) if n_clauses is None else np.asarray(n_clauses, np.int64)
        real = np.arange(nt)[None, :] < n_clauses[:, None]
        df = self.doc_freq(ords)
        uniq, inv = np.unique(df, return_inverse=True)
        w_u = np.array([np.float32(idf(int(d), self.total_num_docs) * (np.float32(1.0) + K1)) for d in uniq], np.float32)
        weights = np.ascontiguousarray(w_u[inv].reshape(nq, nt))
        inner = TopDocs(top_docs.limit + top_docs.offset)
        parts = []
        for s_ord, (seg, o) in enumerate(zip(self.segments, ords)):
            o = np.where(real, o, NO_TERM).astype(np.uint32)
            if mode == MODE_AND:   # a clause this segment cannot satisfy empties its intersection
                dead = ((o == NO_TERM) & real).any(axis=1)
                o[dead] = NO_TERM
            d, sc, n = inner.search_batch(seg, o, mode, weights=weights, average_fieldnorm=self.average_fieldnorm)
            parts.append((s_ord, d, sc, n))
        k = top_docs.limit
        out_seg = np.zeros((nq, k), np.uint32); out_doc = np.zeros((nq, k), np.uint32)
        out_sc = np.zeros((nq, k), np.float32); out_n = np.zeros(nq, np.uint32)
        for q in range(nq):
            segs = np.concatenate([np.full(int(n[q]), s_ord, np.uint32) for s_ord, _, _, n in parts])
            docs = np.concatenate([d[q, :n[q]] for _, d, _, n in parts])
            scs = np.concatenate([sc[q, :n[q]] for _, _, sc, n in parts])
            order = np.lexsort((docs, segs, -scs.astype(np.float64)))[top_docs.offset:top_docs.offset + k]
            m = order.size
            out_seg[q, :m], out_doc[q, :m], out_sc[q, :m], out_n[q] = segs[order], docs[order], scs[order], m
        return out_seg, out_doc, out_sc, out_n

    def search_phrase_batch(self, top_docs, queries_per_segment):
        """queries_per_segment[s] is a list of PhraseQuery in segment s's own ordinals (NO_TERM where the segment does not hold
        the term), the same phrases in the same order for every segment.  The weight of a phrase is Bm25Weight::for_terms over
        the index-wide statistics (doc_freq summed over the segments, terms in offset order); fruits are merged as in
        search_batch.  Returns (segment_ord [nq,k], docs [nq,k], scores [nq,k], n [nq])."""
        nq = len(queries_per_segment[0])
        weights = np.zeros(max(nq, 1), np.float32)
        for q in range(nq):
            dfs = [0] * len(queries_per_segment[0][q].term_ords)
            for seg, qs in zip(self.segments, queries_per_segment):
                for i, t in enumerate(qs[q].term_ords):
                    dfs[i] += int(seg.doc_freq[t]) if t != NO_TERM else 0
            weights[q] = Bm25Weight.for_terms(dfs, self.total_num_docs, self.average_fieldnorm).weight
        inner = TopDocs(top_docs.limit + top_docs.offset)
        parts = []
        for s_ord, (seg, qs) in enumerate(zip(self.segments, queries_per_segment)):
            d, sc, n = inner.search_phrase_batch(seg, qs, weights=weights[:nq], average_fieldnorm=self.average_fieldnorm)
            parts.append((s_ord, d, sc, n))
        k = top_docs.limit
        out_seg = np.zeros((nq, k), np.uint32); out_doc = np.zeros((nq, k), np.uint32)
        out_sc = np.zeros((nq, k), np.float32); out_n = np.zeros(nq, np.uint32)
        for q in range(nq):
            segs = np.concatenate([np.full(int(n[q]), s_ord, np.uint32) for s_ord, _, _, n in parts])
            docs = np.concatenate([d[q, :n[q]] for _, d, _, n in parts])
            scs = np.concatenate([sc[q, :n[q]] for _, _, sc, n in parts])
            order = np.lexsort((docs, segs, -scs.astype(np.float64)))[top_docs.offset:top_docs.offset + k]
            m = order.size
            out_seg[q, :m], out_doc[q, :m], out_sc[q, :m], out_n[q] = segs[order], docs[order], scs[order], m
        return out_seg, out_doc, out_sc, out_n


class SignalComputer:
    """The recall-stage subset of Stract's SignalComputer this path covers: one text field scored with
    Stract's BM25 (coefficient `coeff_text`, e.g. Bm25CleanBody 0.005) plus numeric signal columns
    (coefficient per column), combined in f64 in that order; top-k by (total desc, doc asc)."""

    def __init__(self, segment, signals=None, coefficients=(), coeff_text=0.005, k1=K1, b=B_):
        self.segment, self.signals = segment, signals
        self.coefficients = np.ascontiguousarray(coefficients, np.float64)
        self.coeff_text = float(coeff_text)
        self.k1, self.b = np.float32(k1), np.float32(b)

    def top_docs_batch(self, term_ords, k, max_docs=0, return_stats=False, weights=None, average_fieldnorm=None):
        """`weights` (idf per clause) / `average_fieldnorm` override the segment's own statistics: MultiBm25Weight::for_terms
        takes them from the whole searcher (core/src/ranking/bm25.rs:52-92), see SignalSearcher."""
        seg = self.segment
        term_ords = np.ascontiguousarray(term_ords, np.uint32)
        nq, nt = term_ords.shape
        if weights is None:
            weights = idf_array(seg.doc_freq[np.minimum(term_ords, seg.n_terms - 1)], seg.max_doc)
        weights = np.ascontiguousarray(weights, np.float32)
        cache = compute_tf_cache(seg.average_fieldnorm if average_fieldnorm is None else average_fieldnorm, self.k1, self.b)
        docs = host_out((nq, k), np.uint32); totals = host_out((nq, k), np.float64); n_out = np.zeros(nq, np.uint32)
        sb = B.SignalBatch()
        sb.q = B.Bm25Batch(nq, nt, _p(term_ords), _p(weights), _p(cache), MODE_OR, k)
        sb.k1 = float(self.k1); sb.coeff_text = self.coeff_text
        sb.signals = self.signals._h if self.signals is not None else None
        sb.coeffs = _p(self.coefficients) if self.signals is not None else None
        sb.max_docs = max_docs
        st = B.Bm25Stats()
        check(seg._L.sb200_signal_topk_batch(seg._h, C.byref(sb), _p(docs), _p(totals), _p(n_out), C.byref(st)))
        if return_stats:
            return docs, totals, n_out, {k_: getattr(st, k_) for k_, _ in B.Bm25Stats._fields_ if not k_.startswith("_")}
        return docs, totals, n_out


class SignalSearcher:
    """Path B over several segments: Stract's MultiBm25Weight::for_terms sums total_num_tokens / total_num_docs over the
    segment readers and takes doc_freq from the searcher (core/src/ranking/bm25.rs:52-92); every segment collects its top
    k by `total` and the fruits are merged by (total desc, (segment_ord, doc) asc) like any tantivy top collector
    (tweak_score_top_collector.rs -> TopCollector::merge_fruits, top_collector.rs:109-129)."""

    def __init__(self, computers):
        self.computers = list(computers)          # one SignalComputer per segment (same coefficients)
        segs = [c.segment for c in self.computers]
        self.total_num_docs = int(sum(s.max_doc for s in segs))
        self.total_num_tokens = int(sum(s.total_num_tokens for s in segs))
        self.average_fieldnorm = np.float32(np.float32(self.total_num_tokens) / np.float32(max(self.total_num_docs, 1)))

    def top_docs_batch(self, term_ords_per_segment, k):
        ords = [np.ascontiguousarray(o, np.uint32) for o in term_ords_per_segment]
        nq, nt = ords[0].shape
        df = np.zeros((nq, nt), np.int64)
        for c, o in zip(self.computers, ords):
            seg = c.segment
            df += np.where(o != NO_TERM, seg.doc_freq[np.minimum(o, max(seg.n_terms - 1, 0))].astype(np.int64), 0)
        uniq, inv = np.unique(df, return_inverse=True)
        w_u = np.array([idf(int(d), self.total_num_docs) for d in uniq], np.float32)
        weights = w_u[inv].reshape(nq, nt)
        parts = []
        for s_ord, (c, o) in enumerate(zip(self.computers, ords)):
            # a clause the segment does not hold contributes 0 to every doc: it is dropped, the f32 sum is unchanged
            d, t, n = c.top_docs_batch(o, k, weights=weights, average_fieldnorm=self.average_fieldnorm)
            parts.append((s_ord, d, t, n))
        out_seg = np.zeros((nq, k), np.uint32); out_doc = np.zeros((nq, k), np.uint32)
        out_t = np.zeros((nq, k), np.float64); out_n = np.zeros(nq, np.uint32)
        for q in range(nq):
            segs = np.concatenate([np.full(int(n[q]), s_ord, np.uint32) for s_ord, _, _, n in parts])
            docs = np.concatenate([d[q, :n[q]] for _, d, _, n in parts])
            tot = np.concatenate([t[q, :n[q]] for _, _, t, n in parts])
            order = np.lexsort((docs, segs, -tot))[:k]
            m = order.size
            out_seg[q, :m], out_doc[q, :m], out_t[q, :m], out_n[q] = segs[order], docs[order], tot[order], m
        return out_seg, out_doc, out_t, out_n


# ---- multi-field recall-stage signals (SURVEY 8(f) rank 3) ------------------------------------------------------------
OP_BM25, OP_BM25F, OP_COVERAGE, OP_IDF_SUM, OP_NUMERIC = 0, 1, 2, 3, 4

# The text signals of CoreSignalEnum in declaration order (core/src/ranking/signals/mod.rs:182-206) with what
# SignalComputeOrder::new and prepare_textfields need to know about each: the op kind, its text field (as_field), whether it
# has sibling n-gram signals, and the default coefficient (core/src/ranking/signals/core/text.rs).
CORE_SIGNALS = [
    # name,                                  kind,        field,                              sibling n-grams, default coefficient
    ("Bm25F",                                OP_BM25F,    None,                               False, 0.1),
    ("Bm25Title",                            OP_BM25,     "Title",                            True,  0.0063),
    ("TitleCoverage",                        OP_COVERAGE, "Title",                            False, 0.01),
    ("Bm25TitleBigrams",                     OP_BM25,     "TitleBigrams",                     True,  0.005),
    ("Bm25TitleTrigrams",                    OP_BM25,     "TitleTrigrams",                    True,  0.005),
    ("Bm25CleanBody",                        OP_BM25,     "CleanBody",                        True,  0.005),
    ("CleanBodyCoverage",                    OP_COVERAGE, "CleanBody",                        False, 0.01),
    ("Bm25CleanBodyBigrams",                 OP_BM25,     "CleanBodyBigrams",                 True,  0.005),
    ("Bm25CleanBodyTrigrams",                OP_BM25,     "CleanBodyTrigrams",                True,  0.005),
    ("Bm25StemmedTitle",                     OP_BM25,     "StemmedTitle",                     False, 0.003),
    ("Bm25StemmedCleanBody",                 OP_BM25,     "StemmedCleanBody",                 False, 0.001),
    ("Bm25AllBody",                          OP_BM25,     "AllBody",                          False, 0.0),
    ("Bm25Keywords",                         OP_BM25,     "Keywords",                         False, 0.001),
    ("Bm25BacklinkText",                     OP_BM25,     "BacklinkText",                     False, 0.003),
    ("IdfSumUrl",                            OP_IDF_SUM,  "Url",                              False, 0.0006),
    ("IdfSumSite",                           OP_IDF_SUM,  "SiteWithout",                      False, 0.00015),
    ("IdfSumDomain",                         OP_IDF_SUM,  "Domain",                           False, 0.0003),
    ("IdfSumSiteNoTokenizer",                OP_IDF_SUM,  "SiteNoTokenizer",                  False, 0.00015),
    ("IdfSumDomainNoTokenizer",              OP_IDF_SUM,  "DomainNoTokenizer",                False, 0.0036),
    ("IdfSumDomainNameNoTokenizer",          OP_IDF_SUM,  "DomainNameNoTokenizer",            False, 0.0002),
    ("IdfSumDomainIfHomepage",               OP_IDF_SUM,  "DomainIfHomepage",                 False, 0.0004),
    ("IdfSumDomainNameIfHomepageNoTokenizer", OP_IDF_SUM, "DomainNameIfHomepageNoTokenizer",  False, 0.0036),
    ("IdfSumDomainIfHomepageNoTokenizer",    OP_IDF_SUM,  "DomainIfHomepageNoTokenizer",      False, 0.0036),
    ("IdfSumTitleIfHomepage",                OP_IDF_SUM,  "TitleIfHomepage",                  False, 0.001),
]
# n-gram size and monogram field of the n-gram text fields (core/src/schema/text_field.rs:1267-1403)
NGRAM_FIELDS = {"TitleBigrams": (2, "Title"), "TitleTrigrams": (3, "Title"), "CleanBodyBigrams": (2, "CleanBody"), "CleanBodyTrigrams": (3, "CleanBody")}
# TextFieldEnum declaration order (text_field.rs:161-199), the iteration order of every EnumMap<TextFieldEnum, _>
TEXT_FIELD_ORDER = ["Title", "CleanBody", "StemmedTitle", "StemmedCleanBody", "AllBody", "Url", "UrlNoTokenizer", "UrlForSiteOperator",
                    "SiteWithout", "Domain", "SiteNoTokenizer", "DomainNoTokenizer", "DomainNameNoTokenizer", "SiteIfHomepageNoTokenizer",
                    "DomainIfHomepage", "DomainNameIfHomepageNoTokenizer", "DomainIfHomepageNoTokenizer", "TitleIfHomepage", "BacklinkText",
                    "Description", "DmozDescription", "SchemaOrgJson", "FlattenedSchemaOrgJson", "CleanBodyBigrams", "TitleBigrams",
                    "CleanBodyTrigrams", "TitleTrigrams", "MicroformatTags", "SafetyClassification", "InsertionTimestamp",
                    "RecipeFirstIngredientTagId", "Keywords"]


class SignalComputeOrder:
    """`SignalComputeOrder::new` (core/src/ranking/computer/order.rs:33-62): text signals with sibling n-gram signals are
    grouped per monogram field in an EnumMap (iterated in TextFieldEnum order), each group ordered by descending n-gram
    size (NGramComputeOrder::push re-sorts on every insert); every other signal follows in CoreSignalEnum order.
    `enabled` restricts the list to the signals the caller has fields for; numeric signals (which sit behind the text
    signals in CoreSignalEnum) are appended through `numeric` = [(name, column, coefficient)] in the order given."""

    def __init__(self, enabled, numeric=()):
        groups, others = {}, []
        for name, kind, field, sibling, coef in CORE_SIGNALS:
            if name not in enabled:
                continue
            if sibling:
                ngram, mono = NGRAM_FIELDS.get(field, (1, field))
                groups.setdefault(mono, []).append((ngram, name, kind, field, coef))
                groups[mono].sort(key=lambda e: -e[0])   # sort_unstable_by(b.cmp(a)) on distinct sizes
            else:
                others.append((name, kind, field, coef))
        self.entries = []   # (name, kind, field, chain, col, default coefficient)
        for mono in sorted(groups, key=TEXT_FIELD_ORDER.index):
            for i, (_n, name, kind, field, coef) in enumerate(groups[mono]):
                self.entries.append((name, kind, field, 1 if i == 0 else 2, 0, coef))
        for name, kind, field, coef in others:
            self.entries.append((name, kind, field, 0, 0, coef))
        for name, col, coef in numeric:
            self.entries.append((name, OP_NUMERIC, None, 0, int(col), coef))


class MultiFieldSignalComputer:
    """The recall-stage SignalComputer over several text fields of one segment (core/src/ranking/computer/mod.rs:300-389,
    order.rs): `fields` = {TextField name: SegmentReader} in TextFieldEnum order, every reader opened over the same docs.
    `coefficients` = the query's SignalCoefficients {signal name: coefficient} (`has_query=False`: a SignalComputer built
    without a query), `linear_model` = LinearRegression weights {signal name: weight} (set_linear_model) -- see `coefficient`."""

    def __init__(self, fields, enabled, signals=None, numeric=(), coefficients=None, k1=K1, b=B_, linear_model=None, has_query=True):
        self.names = sorted(fields.keys(), key=TEXT_FIELD_ORDER.index)   # EnumMap<TextFieldEnum, TextFieldData> order
        self.readers = [fields[n] for n in self.names]
        self.signals = signals
        self.order = SignalComputeOrder(set(enabled), numeric)
        self.coefficients = dict(coefficients or {})
        self.linear_model = None if linear_model is None else dict(linear_model)
        self.has_query = bool(has_query)
        self.k1, self.b = np.float32(k1), np.float32(b)
        self._L = lib()

    def coefficient(self, name, default):
        """SignalComputer::coefficient (computer/mod.rs:511-521): with a query, its SignalCoefficients decide -- the entry or
        the signal's default (signals/mod.rs:430-435) -- and the linear model is never asked (`.map(..)` on a Some never
        reaches the `or_else`); without a query the linear model's weight for the signal, else the default."""
        if self.has_query:
            return float(self.coefficients.get(name, default))
        if self.linear_model is not None and name in self.linear_model:
            return float(self.linear_model[name])
        return float(default)

    def field_coefficient(self, field):
        """TextFieldData.signal_coefficient (mod.rs:372): prepare_textfields walks CoreSignalEnum::all() and INSERTS the
        field's data once per signal that names it, so the entry that survives carries the coefficient of the LAST such
        signal (Title ends up with TitleCoverage's, CleanBody with CleanBodyCoverage's)."""
        c = 0.0
        for name, _kind, f, _sib, coef in CORE_SIGNALS:
            if f == field:
                c = self.coefficient(name, coef)
        return c

    def top_docs_batch(self, slot_field, slot_term, k, doc_freq_all_body=None, return_stats=False, slot_boost=None):
        """slot_field / slot_term [n_queries, n_slots]: field index into `self.names` (TextFieldEnum order; 0xFF pads) and the term's ordinal in that
        field's reader (NO_TERM = the segment does not hold it).  idf comes from the field's own doc_freq
        (MultiBm25Weight::for_terms), the Bm25F idf from `doc_freq_all_body` [n_queries, n_slots] (WeightCache: the AllBody
        doc_freq of the token), defaulting to the field's own.  Optic rules: a slot with field | 0x80 is the docset of a rule,
        `slot_boost` [n_queries, n_slots] holds its boost (negative = downrank): SignalComputer::boosts (mod.rs:471-497)."""
        sf = np.ascontiguousarray(slot_field, np.uint8); st = np.ascontiguousarray(slot_term, np.uint32)
        nq, ns = sf.shape
        idf1 = np.zeros((nq, ns), np.float32); idf2 = np.zeros((nq, ns), np.float32)
        dfa_all = None if doc_freq_all_body is None else np.asarray(doc_freq_all_body, np.int64).reshape(nq, ns)
        for f, r in enumerate(self.readers):        # one vectorised pass per field (rule slots and pads keep idf 0)
            m = sf == f
            if not m.any():
                continue
            t = st[m]
            known = (t != NO_TERM) & (t < r.n_terms)
            df = np.zeros(t.shape, np.uint32)
            df[known] = np.asarray(r.doc_freq, np.uint32)[t[known]]
            idf1[m] = idf_array(df, r.max_doc)
            idf2[m] = idf1[m] if dfa_all is None else idf_array(dfa_all[m].astype(np.uint32), r.max_doc)
        caches = [np.ascontiguousarray(compute_tf_cache(r.average_fieldnorm, self.k1, self.b)) for r in self.readers]
        farr = (B.SignalField * len(self.readers))()
        for i, (n_, r) in enumerate(zip(self.names, self.readers)):
            farr[i].seg = r._h; farr[i].tf_cache256 = caches[i].ctypes.data
            farr[i].k1 = float(self.k1); farr[i].bm25f_coefficient = float(np.float32(self.field_coefficient(n_)))
        ops = (B.SignalOp * len(self.order.entries))()
        for i, (name, kind, field, chain, col, coef) in enumerate(self.order.entries):
            ops[i].kind = kind; ops[i].field = self.names.index(field) if field is not None else 0
            ops[i].chain = chain; ops[i].col = col; ops[i].coeff = self.coefficient(name, coef)
        docs = host_out((nq, k), np.uint32); totals = host_out((nq, k), np.float64); n_out = np.zeros(nq, np.uint32)
        mb = B.MultiSignalBatch()
        mb.n_queries, mb.n_slots = nq, ns
        mb.slot_field, mb.slot_term, mb.slot_idf, mb.slot_idf_f = _p(sf), _p(st), _p(idf1), _p(idf2)
        mb.n_fields, mb.n_ops = len(self.readers), len(self.order.entries)
        mb.fields = C.cast(farr, C.c_void_p); mb.ops = C.cast(ops, C.c_void_p)
        mb.signals = self.signals._h if self.signals is not None else None
        mb.k = k
        sbst = None if slot_boost is None else np.ascontiguousarray(slot_boost, np.float64)
        mb.slot_boost = _p(sbst)
        stt = B.Bm25Stats()
        check(self._L.sb200_multi_signal_topk_batch(C.byref(mb), _p(docs), _p(totals), _p(n_out), C.byref(stt)))
        self.last_inputs = dict(idf=idf1, idf_f=idf2, caches=caches)
        if return_stats:
            return docs, totals, n_out, {k_: getattr(stt, k_) for k_, _ in B.Bm25Stats._fields_ if not k_.startswith("_")}
        return docs, totals, n_out
