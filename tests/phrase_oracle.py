"""CPU restatement of tantivy's positions file and slop-0 phrase scoring, the reference the phrase tests check the library
against.  Written from the reference, not from the library: PositionSerializer (positions/serializer.rs), PositionReader::read
(positions/reader.rs), SegmentPostings::positions_with_offset (postings/segment_postings.rs:233-255), PhraseScorer with slop 0
(query/phrase_query/phrase_scorer.rs: compute_phrase_match, intersection, intersection_count, score), Bm25Weight::for_terms
(query/bm25.rs:98-134) and TopDocs' order (score desc, doc asc)."""
import numpy as np

from stract_b200.bm25 import Bm25Weight, compute_tf_cache, fieldnorms_to_ids


def _vint(v):
    out = bytearray()
    while True:
        b = v % 128
        v //= 128
        if v == 0:
            out.append(b | 128)
            return out
        out.append(b)


def _pack4x(block, bits):
    """BitPacker4x::compress: value k in lane k % 4 at slot k // 4, each lane a little-endian bit stream of 32-bit words,
    word w of lane l at u32 index 4 w + l."""
    if bits == 0:
        return b""
    words = np.zeros((bits, 4), np.uint64)
    for lane in range(4):
        acc, fill, w = 0, 0, 0
        for slot in range(32):
            acc |= int(block[slot * 4 + lane]) << fill
            fill += bits
            while fill >= 32:
                words[w, lane] = acc & 0xFFFFFFFF
                acc >>= 32; fill -= 32; w += 1
    return words.astype("<u4").tobytes()


def _unpack4x(data, bits):
    if bits == 0:
        return np.zeros(128, np.uint32)
    words = np.frombuffer(bytes(data[:16 * bits]), "<u4").reshape(bits, 4)
    out = np.zeros(128, np.uint32)
    for lane in range(4):
        stream = 0
        for w in range(bits):
            stream |= int(words[w, lane]) << (32 * w)
        for slot in range(32):
            out[slot * 4 + lane] = (stream >> (slot * bits)) & ((1 << bits) - 1)
    return out


class PositionSerializer:
    def __init__(self):
        self.out = bytearray()
        self.block, self.widths, self.buffer = [], bytearray(), bytearray()

    def write_positions_delta(self, deltas):
        for d in deltas:
            self.block.append(int(d))
            if len(self.block) == 128:
                self._flush_block()

    def _flush_block(self):
        if not self.block:
            return
        if len(self.block) == 128:
            bits = max(self.block).bit_length()        # compress_block_unsorted(.., false)
            self.widths.append(bits)
            self.buffer += _pack4x(self.block, bits)
        else:
            for v in self.block:                        # compress_vint_unsorted
                self.buffer += _vint(v)
        self.block = []

    def close_term(self):
        self._flush_block()
        self.out += _vint(len(self.widths)) + self.widths + self.buffer
        self.widths, self.buffer = bytearray(), bytearray()

    def written_bytes(self):
        return len(self.out)


class PositionReader:
    """PositionReader::open + read(offset, n): the deltas [offset, offset + n) of one term's positions."""

    def __init__(self, data):
        data = bytes(data)
        n, i, sh = 0, 0, 0
        while True:
            b = data[i]; i += 1
            n |= (b & 127) << sh; sh += 7
            if b & 128:
                break
        self.widths = list(data[i:i + n])
        self.blocks_at = []
        p = i + n
        for w in self.widths:
            self.blocks_at.append(p)
            p += 16 * w
        self.data, self.tail_at = data, p
        self._tail, self._blocks = None, {}

    def _block(self, j):
        if j < len(self.widths):
            if j not in self._blocks:
                self._blocks[j] = _unpack4x(self.data[self.blocks_at[j]:], self.widths[j])
            return self._blocks[j]
        if self._tail is None:                          # uncompress_vint_unsorted_until_end
            vals, v, sh = [], 0, 0
            for b in self.data[self.tail_at:]:
                v += (b & 127) << sh; sh += 7
                if b & 128:
                    vals.append(v); v, sh = 0, 0
            self._tail = np.array(vals, np.uint32)
        return self._tail

    def read(self, offset, n):
        out = []
        while n > 0:
            blk = self._block(offset // 128)
            take = blk[offset % 128:offset % 128 + n]
            out.extend(int(x) for x in take)
            offset += len(take); n -= len(take)
            if len(take) == 0:
                raise IndexError("read past the term's positions")
        return np.array(out, np.uint32)


def write_positions(term_tfs, term_positions):
    """Positions file of several terms: (bytes, start[], end[]); term_positions[t] = absolute positions posting by posting."""
    ser = PositionSerializer()
    start, end = [], []
    for tfs, pos in zip(term_tfs, term_positions):
        start.append(ser.written_bytes())
        at = 0
        for tf in tfs:
            p = [int(x) for x in pos[at:at + tf]]
            ser.write_positions_delta([p[0]] + [b - a for a, b in zip(p, p[1:])])   # deltas restart per doc
            at += tf
        ser.close_term()
        end.append(ser.written_bytes())
    return np.frombuffer(bytes(ser.out), np.uint8), np.array(start, np.uint64), np.array(end, np.uint64)


class Index:
    """One segment of one field from whitespace-tokenized texts (or token-id lists): postings (docs, tfs, positions) per term,
    fieldnorm = token count.  `vocab` maps a token to its ordinal (first-seen order unless given)."""

    def __init__(self, docs_tokens, vocab=None):
        self.vocab = dict(vocab or {})
        post = {}
        for d, toks in enumerate(docs_tokens):
            for p, tok in enumerate(toks):
                if tok not in self.vocab:
                    self.vocab[tok] = len(self.vocab)
                post.setdefault(self.vocab[tok], {}).setdefault(d, []).append(p)
        n = len(self.vocab)
        self.term_docs = [np.array(sorted(post.get(t, {})), np.uint32) for t in range(n)]
        self.term_tfs = [np.array([len(post[t][d]) for d in sorted(post.get(t, {}))], np.uint32) for t in range(n)]
        self.term_positions = [np.array([p for d in sorted(post.get(t, {})) for p in post[t][d]], np.uint32) for t in range(n)]
        self.fieldnorms = np.array([len(t) for t in docs_tokens], np.uint32)
        self.fieldnorm_ids = fieldnorms_to_ids(self.fieldnorms)
        self.max_doc = len(docs_tokens)
        self.total_num_tokens = int(self.fieldnorms.sum())
        self.average_fieldnorm = np.float32(np.float32(self.total_num_tokens) / np.float32(max(self.max_doc, 1)))
        self.pos_bytes, self.pos_start, self.pos_end = write_positions(self.term_tfs, self.term_positions)
        self.doc_freq = np.array([len(d) for d in self.term_docs], np.uint32)

    @classmethod
    def from_texts(cls, texts):
        return cls([t.split() for t in texts])

    def positions(self, term, i, shift):
        """positions_with_offset of posting i of `term`: read at Σ tfs[..i] (skip position_offset + the block's freqs before
        the cursor), cumulative sum starting at `shift`, u32."""
        if not hasattr(self, "_readers"):
            self._readers, self._cum = {}, {}
        if term not in self._readers:
            self._readers[term] = PositionReader(self.pos_bytes[int(self.pos_start[term]):int(self.pos_end[term])])
            self._cum[term] = np.concatenate([[0], np.cumsum(self.term_tfs[term].astype(np.uint64))])
        deltas = self._readers[term].read(int(self._cum[term][i]), int(self.term_tfs[term][i]))
        return (np.uint64(shift) + np.cumsum(deltas.astype(np.uint64))).astype(np.uint32)

    def phrase_counts(self, term_ords, offsets=None):
        """{doc: phrase count > 0} of PhraseScorer with slop 0 (the terms as PhraseQuery::new_with_offset sorts them)."""
        offsets = list(range(len(term_ords))) if offsets is None else list(offsets)
        pairs = sorted(zip(offsets, term_ords), key=lambda p: p[0])
        if any(t is None or t >= len(self.term_docs) for _, t in pairs):
            return {}                                   # phrase_scorer() -> None: EmptyScorer
        max_off = max(o for o, _ in pairs)
        # Intersection::new sorts the docsets by size_hint (intersection.rs:68-80)
        sets = sorted([(max_off - o, t) for o, t in pairs], key=lambda st: len(self.term_docs[st[1]]))
        common = set(self.term_docs[sets[0][1]].tolist())
        for _, t in sets[1:]:
            common &= set(self.term_docs[t].tolist())
        out = {}
        for d in sorted(common):
            pos = [self.positions(t, int(np.searchsorted(self.term_docs[t], d)), sh) for sh, t in sets]
            left = pos[0]
            for right in pos[1:-1]:                     # intersection
                left = np.intersect1d(left, right)
                if left.size == 0:
                    break
            count = np.intersect1d(left, pos[-1]).size if left.size else 0   # intersection_count
            if count:
                out[d] = count
        return out

    def weight(self, term_ords, offsets=None, total_num_docs=None, doc_freq=None, avg=None):
        offsets = list(range(len(term_ords))) if offsets is None else list(offsets)
        pairs = sorted(zip(offsets, term_ords), key=lambda p: p[0])
        dfs = [int(self.doc_freq[t]) if doc_freq is None else int(doc_freq[t]) for _, t in pairs]
        return Bm25Weight.for_terms(dfs, self.max_doc if total_num_docs is None else total_num_docs,
                                    self.average_fieldnorm if avg is None else avg)

    def phrase_top_docs(self, term_ords, offsets=None, k=10, weight=None, avg=None):
        """[(score f32, doc)] by (score desc, doc asc)."""
        if any(t is None or t >= len(self.term_docs) for t in term_ords):
            return []
        w = self.weight(term_ords, offsets) if weight is None else weight
        cache = compute_tf_cache(self.average_fieldnorm if avg is None else avg)
        hits = []
        for d, c in self.phrase_counts(term_ords, offsets).items():
            tf = np.float32(c)
            hits.append((np.float32(w.weight * (tf / (tf + cache[self.fieldnorm_ids[d]]))), d))
        hits.sort(key=lambda h: (-float(h[0]), h[1]))
        return hits[:k]
