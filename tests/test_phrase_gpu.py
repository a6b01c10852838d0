"""Phrase queries on the device (sb200_phrase_topk_batch) against the CPU restatement of tantivy's PhraseScorer
(tests/phrase_oracle.py): docs, order and f32 score bits equal.  Random token corpora over a small vocabulary make phrases
match often and terms repeat; long documents put a document's positions across 128-position blocks and into the vint tail,
and frequent terms' posting lists over many blocks."""
import numpy as np
import pytest

import phrase_oracle as O
from stract_b200 import bm25
from stract_b200.bm25 import NO_TERM, PhraseQuery, Searcher, SegmentReader, TopDocs

pytestmark = pytest.mark.gpu

# corpus size and queries per phrase length of test_random_phrases_bit_exact (test_phrase_emulated.py lowers them: the CPU
# emulator runs a warp as 32 coroutines)
RANDOM_DOCS, RANDOM_LEN, QUERIES_PER_LEN = 400, 300, (6, 4, 4)

def _code(name):
    import os
    import re
    txt = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "stract_b200.h")).read()
    return int(re.search(r"#define\s+%s\s+\(?(-?\d+)" % name, txt).group(1))


def segment_of(idx, positions=True, record_option=2):
    data, infos = bm25.encode_postings(idx.term_docs, idx.term_tfs, idx.fieldnorm_ids, idx.average_fieldnorm, record_option=record_option)
    pos = bm25.encode_positions(idx.term_docs, idx.term_tfs, idx.term_positions) if positions else None
    if pos is not None:
        assert np.array_equal(pos[0], idx.pos_bytes)
    return SegmentReader(data, infos, idx.fieldnorm_ids, record_option=record_option, total_num_tokens=idx.total_num_tokens, positions=pos)


def random_index(seed, n_docs, vocab, mean_len, dup_every=0):
    rng = np.random.default_rng(seed)
    p = 1.0 / np.arange(1, vocab + 1); p /= p.sum()
    lens = np.clip(rng.lognormal(np.log(mean_len), 0.8, n_docs), 2, 40 * mean_len).astype(int)
    docs = [list(rng.choice(vocab, n, p=p)) for n in lens]
    if dup_every:
        for d in range(dup_every, n_docs, dup_every):
            docs[d] = list(docs[d - 1])
    return O.Index(docs, vocab={t: t for t in range(vocab)}), rng


def check(idx, seg, queries, k):
    got_d, got_s, got_n = TopDocs.with_limit(k).search_phrase_batch(seg, queries)
    for q, pq in enumerate(queries):
        ords = [None if t == NO_TERM else t for t in pq.term_ords]
        want = idx.phrase_top_docs(ords, pq.offsets, k=k)
        assert int(got_n[q]) == len(want), (q, pq.term_ords, pq.offsets, int(got_n[q]), len(want))
        assert [int(d) for d in got_d[q, :got_n[q]]] == [d for _, d in want], (q, pq.term_ords, pq.offsets)
        assert np.array_equal(got_s[q, :got_n[q]].view(np.uint32), np.array([s for s, _ in want], np.float32).view(np.uint32)), q


def test_reference_scenarios_on_device():
    cases = [
        (["b b b d c g c", "a b b d c g c", "a b a b c", "c a b a d ga a", "a b c"],
         [["a", "b"], ["a", "b", "c"], ["b", "b"], ["g", "ewrwer"], ["g", "a"]], None),
        (["b", "a b", "b a"], [["a", "b"], ["b", "a"]], None),
        (["a b c d e f g h"], [["a", "b"], ["b", "a"], ["a", "b"], ["a", "c"], ["a", "c", "d"], ["a", "c", "e"], ["e", "a", "c"], ["a", "d"], ["a", "c"]],
         [[0, 1], [1, 0], [0, 2], [0, 2], [0, 2, 3], [0, 2, 4], [4, 0, 2], [0, 2], [1, 3]]),
        (["a c", "a a b d a b c", " a b"], [["a", "b"]], None),
        (["a b c", "a b c a b"], [["a", "b"]], None),
    ]
    for texts, phrases, offsets in cases:
        idx = O.Index.from_texts(texts)
        seg = segment_of(idx)
        qs = [PhraseQuery([idx.vocab.get(w, NO_TERM) for w in ph], None if offsets is None else offsets[i]) for i, ph in enumerate(phrases)]
        check(idx, seg, qs, 10)
        seg.close()
    idx = O.Index.from_texts(["a b c", "a b c a b"])
    seg = segment_of(idx)
    _, s, _ = TopDocs.with_limit(10).search_phrase_batch(seg, [PhraseQuery([idx.vocab["a"], idx.vocab["b"]])])
    assert [int(x) for x in s[0, :2].view(np.uint32)] == [0x3EEFD840, 0x3ECFF775]   # test_oracle_phrase.PHRASE_SCORE
    seg.close()


def random_queries(rng, idx, n, lens, vocab):
    qs = []
    for i in range(n):
        L = int(lens[i % len(lens)])
        terms = [int(x) for x in rng.integers(0, vocab, L)]
        offs = list(range(L))
        if i % 4 == 1:
            offs = sorted(int(x) for x in rng.choice(3 * L, L, replace=False))
            offs = [o + 2 for o in offs]
            perm = rng.permutation(L)
            terms = [terms[j] for j in perm]; offs = [offs[j] for j in perm]
        if i % 5 == 2:
            terms[1] = terms[0]
        qs.append(PhraseQuery(terms, offs))
    return qs


def phrases_from_docs(rng, docs, n, L, gaps=False):
    qs = []
    for _ in range(n):
        d = docs[int(rng.integers(len(docs)))]
        while len(d) < 3 * L + 3:
            d = docs[int(rng.integers(len(docs)))]
        at = int(rng.integers(0, len(d) - 3 * L - 2))
        offs = sorted(int(x) for x in rng.choice(3 * L, L, replace=False)) if gaps else list(range(L))
        terms = [int(d[at + o]) for o in offs]
        perm = rng.permutation(L)
        qs.append(PhraseQuery([terms[j] for j in perm], [offs[j] + (5 if gaps else 0) for j in perm]))
    return qs


def test_random_phrases_bit_exact():
    idx, rng = random_index(11, RANDOM_DOCS, 12, RANDOM_LEN)
    toks = {}
    for t in range(len(idx.term_docs)):
        at = 0
        for d, tf in zip(idx.term_docs[t], idx.term_tfs[t]):
            for p in idx.term_positions[t][at:at + tf]:
                toks.setdefault(int(d), {})[int(p)] = t
            at += tf
    docs = [[toks[d][p] for p in sorted(toks[d])] for d in range(idx.max_doc)]
    seg = segment_of(idx)
    assert seg.info()["hbm_bytes"] > idx.pos_bytes.size
    assert max(len(x) for x in idx.term_docs) > 2 * 128 and int(idx.term_tfs[0].max()) > 128
    a, b, c = QUERIES_PER_LEN
    for L in range(2, 9):
        qs = phrases_from_docs(rng, docs, a, L) + phrases_from_docs(rng, docs, b, L, gaps=True) + random_queries(rng, idx, c, [L], 12)
        check(idx, seg, qs, 50)
    mixed = phrases_from_docs(rng, docs, 5, 2) + phrases_from_docs(rng, docs, 5, 5, gaps=True) + [PhraseQuery([0, 0]), PhraseQuery([3, 3, 3], [0, 2, 1])]
    for k in (1, 7, 1000):
        check(idx, seg, mixed, k)
    check(idx, seg, [PhraseQuery([1, NO_TERM, 2]), PhraseQuery([NO_TERM, 1])] + mixed[:3], 100)
    _, _, _, st = TopDocs.with_limit(10).search_phrase_batch(seg, mixed[:2], return_stats=True)
    assert st["postings_scored"] == sum(int(idx.doc_freq[t]) for q in mixed[:2] for t in q.term_ords) and st["docs_scored"] > 0
    seg.close()


def test_ties_order_by_doc():
    idx, rng = random_index(5, 200, 6, 40, dup_every=2)
    seg = segment_of(idx)
    check(idx, seg, [PhraseQuery([0, 1]), PhraseQuery([1, 0, 2]), PhraseQuery([2, 2])], 30)
    seg.close()


def test_searcher_over_three_segments_matches_one_big_segment():
    idx, rng = random_index(23, 300, 10, 120)
    docs_tok = {}
    for t in range(len(idx.term_docs)):
        at = 0
        for d, tf in zip(idx.term_docs[t], idx.term_tfs[t]):
            for p in idx.term_positions[t][at:at + tf]:
                docs_tok.setdefault(int(d), {})[int(p)] = t
            at += tf
    docs = [[docs_tok[d][p] for p in sorted(docs_tok[d])] for d in range(idx.max_doc)]
    cuts = [0, 90, 200, 300]
    parts = [O.Index(docs[a:b], vocab={t: t for t in range(10)}) for a, b in zip(cuts, cuts[1:])]
    segs = [segment_of(p) for p in parts]
    big = segment_of(idx)
    qs = phrases_from_docs(rng, docs, 12, 2) + phrases_from_docs(rng, docs, 8, 3, gaps=True)
    per_seg = []
    for p in parts:
        per_seg.append([PhraseQuery([t if p.doc_freq[t] else NO_TERM for t in q.term_ords], q.offsets) for q in qs])
    s_ord, s_doc, s_sc, s_n = Searcher(segs).search_phrase_batch(TopDocs.with_limit(40), per_seg)
    b_doc, b_sc, b_n = TopDocs.with_limit(40).search_phrase_batch(big, qs)
    assert np.array_equal(s_n, b_n)
    for q in range(len(qs)):
        glob = np.array([cuts[s] + d for s, d in zip(s_ord[q, :s_n[q]], s_doc[q, :s_n[q]])], np.uint32)
        assert np.array_equal(glob, b_doc[q, :b_n[q]]), q
        assert np.array_equal(s_sc[q, :s_n[q]].view(np.uint32), b_sc[q, :b_n[q]].view(np.uint32)), q
    for s in segs + [big]:
        s.close()


def test_term_info_store_positions_ranges_on_device():
    import oracle
    n = 1000
    off = lambda i: i * 13 + i * i   # noqa: E731
    ps = np.array([off(i) for i in range(n)], np.uint64); pe = np.array([off(i + 1) for i in range(n)], np.uint64)
    qs = np.array([7 * i * i for i in range(n)], np.uint64); qe = np.array([7 * (i + 1) * (i + 1) for i in range(n)], np.uint64)
    store = oracle.term_info_store_write(np.arange(n, dtype=np.uint32), ps, pe, qs, qe)
    infos, cnt, (gs, ge) = bm25.decode_term_info_store(store, with_positions=True)
    assert cnt == n
    want = [oracle.term_info_store_get(store, i)[3:] for i in range(n)]
    assert [(int(a), int(b)) for a, b in zip(gs, ge)] == want
    # a real segment opened from its TermInfoStore with positions
    idx, rng = random_index(3, 150, 8, 60)
    data, tinfo = bm25.encode_postings(idx.term_docs, idx.term_tfs, idx.fieldnorm_ids, idx.average_fieldnorm, record_option=2)
    t_off = np.array([tinfo[i].postings_off for i in range(len(idx.term_docs))], np.uint64)
    t_len = np.array([tinfo[i].postings_len for i in range(len(idx.term_docs))], np.uint64)
    store = oracle.term_info_store_write(idx.doc_freq, t_off, t_off + t_len, idx.pos_start, idx.pos_end)
    infos, cnt, pos = bm25.decode_term_info_store(store, with_positions=True)
    seg = SegmentReader(data, infos, idx.fieldnorm_ids, record_option=2, total_num_tokens=idx.total_num_tokens, positions=(idx.pos_bytes, *pos))
    check(idx, seg, [PhraseQuery([0, 1]), PhraseQuery([2, 0, 1])], 20)
    seg.close()


def _rc(fn):
    from stract_b200._lib import Sb200Error
    try:
        fn()
    except Sb200Error as e:
        return e.code
    return 0


def test_errors():
    idx = O.Index.from_texts(["a b c", "a b c a b"] * 100)
    seg = segment_of(idx, positions=False)
    assert _rc(lambda: TopDocs.with_limit(5).search_phrase_batch(seg, [PhraseQuery([0, 1])])) == _code("SB200_EINVAL")
    seg.close()
    seg1 = segment_of(idx, positions=False, record_option=1)
    assert _rc(lambda: seg1.attach_positions(idx.pos_bytes, idx.pos_start, idx.pos_end)) == _code("SB200_EINVAL")
    seg1.close()
    seg = segment_of(idx)
    bad = PhraseQuery([0, 1]); bad.term_ords, bad.offsets = [0], [0]
    assert _rc(lambda: TopDocs.with_limit(5).search_phrase_batch(seg, [PhraseQuery([0, 1]), bad])) == _code("SB200_EINVAL")
    seg.close()
    # corrupt positions -> SB200_EFORMAT at attach
    t = int(np.argmax([int(x.sum()) for x in idx.term_tfs]))    # a term with full 128-position blocks
    assert int(idx.term_tfs[t].sum()) >= 128
    s0, e0 = int(idx.pos_start[t]), int(idx.pos_end[t])
    truncated = idx.pos_end.copy(); truncated[t] = e0 - 1
    wide = idx.pos_bytes.copy(); wide[s0 + 1] = 33                  # the first bit width (VInt(#blocks) is one byte here)
    count = idx.pos_bytes.copy(); count[s0] = (idx.pos_bytes[s0] & 0x7F) + 1 | 0x80
    outside = idx.pos_end.copy(); outside[t] = idx.pos_bytes.size + 5
    for data, ps, pe in [(idx.pos_bytes, idx.pos_start, truncated), (wide, idx.pos_start, idx.pos_end), (count, idx.pos_start, idx.pos_end),
                         (idx.pos_bytes, idx.pos_start, outside)]:
        s = segment_of(idx, positions=False)
        assert _rc(lambda: s.attach_positions(data, ps, pe)) == _code("SB200_EFORMAT")
        assert _rc(lambda: TopDocs.with_limit(5).search_phrase_batch(s, [PhraseQuery([0, 1])])) == _code("SB200_EINVAL")
        s.close()
