"""The phrase oracle (tests/phrase_oracle.py) pinned on the reference's own tests -- positions/mod.rs:85-238 and
query/phrase_query/{mod.rs, phrase_weight.rs:113-135} -- and the library's positions writer checked byte for byte against it."""
import numpy as np

import phrase_oracle as O


def _file(deltas):
    ser = O.PositionSerializer()
    ser.write_positions_delta(deltas)
    ser.close_term()
    return bytes(ser.out)


def test_position_file_sizes_and_reads():
    data = _file(range(1000))
    assert len(data) == 1224
    r = O.PositionReader(data)
    assert list(r.read(0, 1000)) == list(range(1000))
    for offset in range(0, 1000, 37):
        assert list(r.read(offset, min(50, 1000 - offset))) == list(range(offset, min(offset + 50, 1000)))
    data = _file(range(512))
    assert len(data) == 533
    r = O.PositionReader(data)
    assert r.read(230, 1)[0] == 230 and r.read(9, 1)[0] == 9
    assert len(_file(range(2_000_000))) == 5_003_499
    r = O.PositionReader(_file(range(2_000_000)))
    assert list(r.read(128, 256)) == list(range(128, 384))
    assert r.read(1_999_999, 1)[0] == 1_999_999
    data = _file([9] * 2_000_000)
    assert len(data) == 1_015_627
    assert O.PositionReader(data).read(0, 1)[0] == 9
    assert _file([]) == bytes([0x80])                  # test_empty_position: VInt(0)
    ser = O.PositionSerializer()                       # test_multiple_write_positions
    ser.write_positions_delta([1, 12]); ser.write_positions_delta([4, 17]); ser.write_positions_delta([443])
    ser.close_term()
    assert list(O.PositionReader(bytes(ser.out)).read(0, 5)) == [1, 12, 4, 17, 443]


def _top(idx, words, offsets=None):
    ords = [idx.vocab.get(w) for w in words]
    return [d for _, d in idx.phrase_top_docs(ords, offsets, k=100)]


def test_phrase_query():
    idx = O.Index.from_texts(["b b b d c g c", "a b b d c g c", "a b a b c", "c a b a d ga a", "a b c"])
    assert sorted(_top(idx, ["a", "b"])) == [1, 2, 3, 4]
    assert sorted(_top(idx, ["a", "b", "c"])) == [2, 4]
    assert sorted(_top(idx, ["b", "b"])) == [0, 1]
    assert _top(idx, ["g", "ewrwer"]) == []
    assert _top(idx, ["g", "a"]) == []


def test_phrase_query_docfreq_order():
    idx = O.Index.from_texts(["b", "a b", "b a"])
    assert _top(idx, ["a", "b"]) == [1]
    assert _top(idx, ["b", "a"]) == [2]


def test_phrase_query_non_trivial_offsets():
    idx = O.Index.from_texts(["a b c d e f g h"])
    q = lambda pairs: _top(idx, [w for _, w in pairs], [o for o, _ in pairs])  # noqa: E731
    assert q([(0, "a"), (1, "b")]) == [0]
    assert q([(1, "b"), (0, "a")]) == [0]
    assert q([(0, "a"), (2, "b")]) == []
    assert q([(0, "a"), (2, "c")]) == [0]
    assert q([(0, "a"), (2, "c"), (3, "d")]) == [0]
    assert q([(0, "a"), (2, "c"), (4, "e")]) == [0]
    assert q([(4, "e"), (0, "a"), (2, "c")]) == [0]
    assert q([(0, "a"), (2, "d")]) == []
    assert q([(1, "a"), (3, "c")]) == [0]


def test_phrase_count():
    idx = O.Index.from_texts(["a c", "a a b d a b c", " a b"])
    assert idx.phrase_counts([idx.vocab["a"], idx.vocab["b"]]) == {1: 2, 2: 1}


# The reference asserts these to assert_nearly_equals (relative 5e-5; its test lists them in doc order).  The f32 bits this
# restatement computes are recorded as well: the GPU path must reproduce them exactly.
PHRASE_SCORE = {0: (0.40618482, 0x3ECFF775), 1: (0.46844664, 0x3EEFD840)}


def test_phrase_score():
    idx = O.Index.from_texts(["a b c", "a b c a b"])
    got = idx.phrase_top_docs([idx.vocab["a"], idx.vocab["b"]], k=10)
    assert [d for _, d in got] == [1, 0]
    for s, d in got:
        want, bits = PHRASE_SCORE[d]
        assert abs(float(s) - want) <= 5e-5 * want
        assert int(np.float32(s).view(np.uint32)) == bits


def _random_terms(rng, n_terms, max_doc):
    docs, tfs, pos = [], [], []
    for npos in n_terms:
        # a term with exactly npos positions over random docs
        per = []
        left = npos
        while left:
            tf = int(min(left, rng.integers(1, 40)))
            per.append(tf); left -= tf
        d = np.sort(rng.choice(max_doc, len(per), replace=False)).astype(np.uint32)
        t = np.array(per, np.uint32)
        p = np.concatenate([np.sort(rng.choice(5000, tf, replace=False)) for tf in per]).astype(np.uint32) if per else np.zeros(0, np.uint32)
        docs.append(d); tfs.append(t); pos.append(p)
    return docs, tfs, pos


def test_library_writer_matches_oracle_writer():
    from stract_b200 import bm25
    rng = np.random.default_rng(7)
    counts = [0, 1, 127, 128, 129, 255, 256, 1000, 4097]
    docs, tfs, pos = _random_terms(rng, counts, 3000)
    want, ws, we = O.write_positions(tfs, pos)
    got, gs, ge = bm25.encode_positions(docs, tfs, pos, threads=3)
    assert np.array_equal(got, want) and np.array_equal(gs, ws) and np.array_equal(ge, we)
    for t, n in enumerate(counts):
        r = O.PositionReader(got[int(gs[t]):int(ge[t])])
        if n:
            deltas = r.read(0, n)
            at = 0
            for tf in tfs[t]:
                assert np.array_equal(np.cumsum(deltas[at:at + tf]), pos[t][at:at + tf]); at += tf


def test_term_info_store_oracle_positions_ranges():
    """The oracle's TermInfoStore writer/reader round-trips positions ranges (the device decoder is checked against it in
    test_phrase_gpu.py)."""
    import oracle
    n = 1000
    off = lambda i: i * 13 + i * i   # noqa: E731
    ps = np.array([off(i) for i in range(n)], np.uint64); pe = np.array([off(i + 1) for i in range(n)], np.uint64)
    qs = np.array([7 * i * i for i in range(n)], np.uint64); qe = np.array([7 * (i + 1) * (i + 1) for i in range(n)], np.uint64)
    store = oracle.term_info_store_write(np.arange(n, dtype=np.uint32), ps, pe, qs, qe)
    want = [oracle.term_info_store_get(store, i)[3:] for i in range(n)]
    assert want == [(int(a), int(b)) for a, b in zip(qs, qe)]
