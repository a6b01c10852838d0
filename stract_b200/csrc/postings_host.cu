// postings_host.cu -- host-side (CPU) writer of tantivy-format posting lists.
//
// Builds synthetic / test segments in the exact byte format the device decoder consumes:
//   [VInt skip_len][skip entries][blocks ...][vint tail]          (skip section only when doc_freq >= 128)
//   block  = 128 strict-delta doc ids bit-packed (BitPacker4x layout), then 128 (tf-1) bit-packed
//   skip   = last_doc u32 LE | 0x40+doc_bits | tf_bits | blockwand fieldnorm_id | blockwand tf (255 = inf)
//   tail   = doc deltas then tfs, 7 bits per byte, stop bit (0x80) on the LAST byte of a value
// Reference: tantivy/src/postings/serializer.rs:343-462, skip.rs:13-76, compression/{mod.rs:33-74,vint.rs}.
// BitPacker4x (crate `bitpacking` 0.9.2, not in /root/reference): 4 interleaved lanes, value k in lane k&3
// at slot k>>2, lane streams little-endian over 32-bit words, word w of lane l at u32 index 4w+l.
#include "common.cuh"
#include "../../include/stract_b200_bm25.h"

#include <algorithm>
#include <cmath>
#include <thread>
#include <vector>

namespace sb200 {

// fieldnorm byte code: identity below 24, then 3 mantissa bits + exponent (fieldnorm/code.rs:298-318)
uint32_t fieldnorm_value(uint8_t id) {
  if (id < 24) return id;
  const uint32_t x = id - 24u, mant = x & 7u, ex = x >> 3;
  return 24u + (ex == 0 ? mant : ((mant | 8u) << (ex - 1)));
}
uint8_t fieldnorm_id(uint32_t v) {
  int lo = 0, hi = 255;  // largest id with value(id) <= v
  while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (fieldnorm_value((uint8_t)mid) <= v) lo = mid; else hi = mid - 1; }
  return (uint8_t)lo;
}

namespace {

inline int width_of(uint32_t orred) { return orred ? 32 - __builtin_clz(orred) : 0; }

// appends the 4-lane interleaved packing of 128 values at `w` bits each
void pack4x(const uint32_t* v, int w, std::vector<uint8_t>& out) {
  if (w == 0) return;
  const size_t at = out.size();
  out.resize(at + (size_t)w * 16, 0);
  uint32_t* dst = reinterpret_cast<uint32_t*>(out.data() + at);  // appended region; alignment handled by memcpy below
  std::vector<uint32_t> tmp((size_t)w * 4, 0u);
  for (int lane = 0; lane < 4; lane++) {
    uint64_t acc = 0; int fill = 0; int word = 0;
    for (int slot = 0; slot < 32; slot++) {
      const uint64_t x = (w == 32) ? v[slot * 4 + lane] : (v[slot * 4 + lane] & ((1u << w) - 1u));
      acc |= x << fill; fill += w;
      while (fill >= 32) { tmp[(size_t)word * 4 + lane] = (uint32_t)acc; acc >>= 32; fill -= 32; word++; }
    }
  }
  (void)dst;
  memcpy(out.data() + at, tmp.data(), tmp.size() * 4);
}

void put_vint(std::vector<uint8_t>& out, uint64_t v) {
  while (v >= 128) { out.push_back((uint8_t)(v & 127)); v >>= 7; }
  out.push_back((uint8_t)v | 0x80);
}

struct TermBytes { std::vector<uint8_t> bytes; };

// tantivy Bm25Weight pieces needed for the block-wand (fieldnorm_id, tf) pair: only tf/(tf+norm) matters
struct TfNorm {
  float norm[256];
  explicit TfNorm(float avg) { for (int i = 0; i < 256; i++) norm[i] = 1.2f * (1.0f - 0.75f + 0.75f * (float)fieldnorm_value((uint8_t)i) / avg); }
  float factor(uint8_t id, uint32_t tf) const { const float t = (float)tf; return t / (t + norm[id]); }
};

// record: 1 = IndexRecordOption::WithFreqs (8-byte skip entries), 2 = WithFreqsAndPositions (12 bytes: the sum of the
// block's term freqs sits between tf_bits and the block-wand pair, skip.rs:52-76; positions live in another file)
void encode_term(const uint32_t* docs, const uint32_t* tfs, uint32_t df, const uint8_t* fn_ids, bool have_fn,
                 const TfNorm& tn, int record, std::vector<uint8_t>& out) {
  std::vector<uint8_t> skip, body;
  const uint32_t full = df / 128;
  uint32_t prev = 0;
  uint32_t delta[128], tfm1[128];
  for (uint32_t b = 0; b < full; b++) {
    const uint32_t* d = docs + (size_t)b * 128; const uint32_t* t = tfs + (size_t)b * 128;
    uint32_t run = (prev == 0) ? 0xFFFFFFFFu : prev;  // offset 0 means "no previous doc": first value stored verbatim
    uint32_t ord = 0, ort = 0;
    for (int i = 0; i < 128; i++) { delta[i] = d[i] - run - 1u; run = d[i]; ord |= delta[i]; tfm1[i] = t[i] - 1u; ort |= tfm1[i]; }
    const int wd = width_of(ord), wt = width_of(ort);
    pack4x(delta, wd, body);
    pack4x(tfm1, wt, body);
    prev = d[127];
    for (int i = 0; i < 4; i++) skip.push_back((uint8_t)(prev >> (8 * i)));
    skip.push_back((uint8_t)(wd | 0x40));
    skip.push_back((uint8_t)wt);
    if (record == 2) {  // write_total_term_freq, serializer.rs:383-388
      uint32_t sum = 0;
      for (int i = 0; i < 128; i++) sum += t[i];
      for (int i = 0; i < 4; i++) skip.push_back((uint8_t)(sum >> (8 * i)));
    }
    uint8_t bid = 0; uint32_t btf = 0;
    if (have_fn) {  // Iterator::max_by keeps the last of equal maxima
      float best = 0; bool any = false;
      for (int i = 0; i < 128; i++) {
        const uint8_t id = fn_ids[d[i]]; const float f = tn.factor(id, t[i]);
        if (!any || f >= best) { best = f; bid = id; btf = t[i]; any = true; }
      }
    }
    skip.push_back(bid);
    skip.push_back((uint8_t)std::min<uint32_t>(btf, 255u));
  }
  const uint32_t rest = df - full * 128;
  uint32_t run = prev;
  for (uint32_t i = 0; i < rest; i++) { const uint32_t x = docs[(size_t)full * 128 + i]; put_vint(body, x - run); run = x; }
  for (uint32_t i = 0; i < rest; i++) put_vint(body, tfs[(size_t)full * 128 + i]);
  if (df >= 128) { put_vint(out, skip.size()); out.insert(out.end(), skip.begin(), skip.end()); }
  out.insert(out.end(), body.begin(), body.end());
}

// PositionSerializer::write_positions_delta + close_term for one term (tantivy/src/positions/serializer.rs, format in
// positions/mod.rs:7-30): VInt(#full blocks), one bit width per block, the blocks (BitPacker4x, unsorted, not minus-one
// encoded: compression/mod.rs:51-67), then the P % 128 remaining deltas as unsorted vints (compression/vint.rs:24-42).
// `pos` holds the term's Σtf absolute positions posting by posting; a document's first delta is its first position
// (postings/serializer.rs:191-205).  Returns false when a document's positions are not strictly ascending.
bool encode_positions_term(const uint32_t* tfs, uint32_t df, const uint32_t* pos, std::vector<uint8_t>& out) {
  std::vector<uint32_t> delta;
  uint64_t n = 0;
  for (uint32_t i = 0; i < df; i++) n += tfs[i];
  delta.resize(n);
  uint64_t at = 0;
  for (uint32_t i = 0; i < df; i++) {
    uint32_t prev = 0;
    for (uint32_t j = 0; j < tfs[i]; j++, at++) {
      if (j && pos[at] <= prev) return false;
      delta[at] = pos[at] - prev; prev = pos[at];
    }
  }
  const uint64_t nb = n / 128;
  std::vector<uint8_t> widths(nb), body;
  for (uint64_t b = 0; b < nb; b++) {
    uint32_t orred = 0;
    for (int i = 0; i < 128; i++) orred |= delta[b * 128 + i];
    widths[b] = (uint8_t)width_of(orred);
    pack4x(delta.data() + b * 128, widths[b], body);
  }
  for (uint64_t i = nb * 128; i < n; i++) put_vint(body, delta[i]);
  put_vint(out, nb);
  out.insert(out.end(), widths.begin(), widths.end());
  out.insert(out.end(), body.begin(), body.end());
  return true;
}

}  // namespace
}  // namespace sb200

extern "C" {

uint32_t sb200_fieldnorm_id_to_value(uint8_t id) { return sb200::fieldnorm_value(id); }
uint8_t sb200_fieldnorm_value_to_id(uint32_t v) { return sb200::fieldnorm_id(v); }

// idf of tantivy/src/query/bm25.rs:52-56 == core/src/ranking/bm25.rs:23-27 for a whole array of doc_freqs, in f32 with the C
// library's logf (what Rust's f32::ln lowers to on Linux); tantivy_weight != 0 multiplies by (1 + K1) like Bm25Weight
// (bm25.rs:161-162).  Host code: a batch's weights no longer cost one interpreter round trip per distinct doc_freq.
int sb200_bm25_idf(const uint32_t* doc_freq, uint64_t n, uint64_t doc_count, int tantivy_weight, float* out) {
  if ((n && (!doc_freq || !out))) { sb200::set_error("NULL argument"); return SB200_EINVAL; }
  for (uint64_t i = 0; i < n; i++) {
    if (doc_freq[i] > doc_count) { sb200::set_error("doc_freq %u > doc_count %llu", doc_freq[i], (unsigned long long)doc_count); return SB200_EINVAL; }
    const volatile float x = ((float)(doc_count - doc_freq[i]) + 0.5f) / ((float)doc_freq[i] + 0.5f);
    const volatile float l = logf(1.0f + x);
    out[i] = tantivy_weight ? l * (1.0f + 1.2f) : l;
  }
  return SB200_OK;
}

int sb200_postings_encode(const uint32_t* docs, const uint32_t* tfs, const uint64_t* term_off, uint32_t n_terms,
                          const uint8_t* fieldnorm_ids, uint32_t max_doc, float avg_fieldnorm, uint8_t* out,
                          uint64_t out_cap, uint64_t* out_len, sb200_term_info* infos, int threads) {
  return sb200_postings_encode_ex(docs, tfs, term_off, n_terms, fieldnorm_ids, max_doc, avg_fieldnorm, 1, out, out_cap, out_len,
                                  infos, threads);
}

int sb200_postings_encode_ex(const uint32_t* docs, const uint32_t* tfs, const uint64_t* term_off, uint32_t n_terms,
                             const uint8_t* fieldnorm_ids, uint32_t max_doc, float avg_fieldnorm, int record_option,
                             uint8_t* out, uint64_t out_cap, uint64_t* out_len, sb200_term_info* infos, int threads) {
  using namespace sb200;
  if (!term_off || !out_len || (n_terms && (!docs || !tfs))) SB_FAIL(SB200_EINVAL, "NULL argument");
  if (record_option != 1 && record_option != 2) SB_FAIL(SB200_EINVAL, "record_option %d: the writer covers WithFreqs (1) and WithFreqsAndPositions (2)", record_option);
  const bool have_fn = fieldnorm_ids != nullptr && max_doc > 0;
  const TfNorm tn(avg_fieldnorm);
  std::vector<TermBytes> enc(n_terms);
  std::atomic<uint32_t> next(0);
  std::atomic<int> bad(0);
  auto work = [&]() {
    for (;;) {
      const uint32_t t = next.fetch_add(64);
      if (t >= n_terms) break;
      for (uint32_t u = t; u < std::min(n_terms, t + 64); u++) {
        const uint64_t a = term_off[u], b = term_off[u + 1];
        if (b < a || b - a > 0x7FFFFFFFull) { bad = 1; continue; }
        const uint32_t df = (uint32_t)(b - a);
        for (uint32_t i = 0; i < df; i++) {
          if (tfs[a + i] == 0 || (i && docs[a + i] <= docs[a + i - 1]) || (have_fn && docs[a + i] >= max_doc)) { bad = 1; break; }
        }
        if (!bad) encode_term(docs + a, tfs + a, df, fieldnorm_ids, have_fn, tn, record_option, enc[u].bytes);
      }
    }
  };
  const int nt = std::max(1, threads);
  std::vector<std::thread> pool;
  for (int i = 0; i < nt; i++) pool.emplace_back(work);
  for (auto& th : pool) th.join();
  if (bad) SB_FAIL(SB200_EINVAL, "posting input must be ascending doc ids < max_doc with tf >= 1");
  uint64_t total = 0;
  for (uint32_t t = 0; t < n_terms; t++) total += enc[t].bytes.size();
  *out_len = total;
  if (!out) return SB200_OK;
  if (out_cap < total) SB_FAIL(SB200_EINVAL, "output buffer too small: need %llu bytes", (unsigned long long)total);
  uint64_t at = 0;
  for (uint32_t t = 0; t < n_terms; t++) {
    if (infos) { infos[t].postings_off = at; infos[t].postings_len = enc[t].bytes.size(); infos[t].doc_freq = (uint32_t)(term_off[t + 1] - term_off[t]); infos[t]._pad = 0; }
    memcpy(out + at, enc[t].bytes.data(), enc[t].bytes.size());
    at += enc[t].bytes.size();
  }
  return SB200_OK;
}

int sb200_positions_encode(const uint32_t* docs, const uint32_t* tfs, const uint64_t* term_off, uint32_t n_terms,
                           const uint32_t* positions, uint8_t* out, uint64_t out_cap, uint64_t* out_len, uint64_t* pos_start,
                           uint64_t* pos_end, int threads) {
  using namespace sb200;
  if (!term_off || !out_len || (n_terms && (!docs || !tfs || !positions))) SB_FAIL(SB200_EINVAL, "NULL argument");
  // positions of posting i of term t start at Σ tfs[..i] over the whole CSR
  std::vector<uint64_t> pos_off(n_terms + 1, 0);
  for (uint32_t t = 0; t < n_terms; t++) {
    const uint64_t a = term_off[t], b = term_off[t + 1];
    if (b < a || b - a > 0x7FFFFFFFull) SB_FAIL(SB200_EINVAL, "term %u: term_off is not ascending", t);
    uint64_t s = 0;
    for (uint64_t i = a; i < b; i++) s += tfs[i];
    pos_off[t + 1] = pos_off[t] + s;
  }
  std::vector<TermBytes> enc(n_terms);
  std::atomic<uint32_t> next(0);
  std::atomic<int> bad(0);
  auto work = [&]() {
    for (;;) {
      const uint32_t t = next.fetch_add(64);
      if (t >= n_terms) break;
      for (uint32_t u = t; u < std::min(n_terms, t + 64); u++) {
        const uint64_t a = term_off[u];
        const uint32_t df = (uint32_t)(term_off[u + 1] - a);
        for (uint32_t i = 0; i < df; i++) if (tfs[a + i] == 0 || (i && docs[a + i] <= docs[a + i - 1])) { bad = 1; break; }
        if (!bad && !encode_positions_term(tfs + a, df, positions + pos_off[u], enc[u].bytes)) bad = 2;
      }
    }
  };
  const int nt = std::max(1, threads);
  std::vector<std::thread> pool;
  for (int i = 0; i < nt; i++) pool.emplace_back(work);
  for (auto& th : pool) th.join();
  if (bad == 1) SB_FAIL(SB200_EINVAL, "posting input must be ascending doc ids with tf >= 1");
  if (bad == 2) SB_FAIL(SB200_EINVAL, "the positions of a document must be strictly ascending");
  uint64_t total = 0;
  for (uint32_t t = 0; t < n_terms; t++) total += enc[t].bytes.size();
  *out_len = total;
  if (!out) return SB200_OK;
  if (out_cap < total) SB_FAIL(SB200_EINVAL, "output buffer too small: need %llu bytes", (unsigned long long)total);
  uint64_t at = 0;
  for (uint32_t t = 0; t < n_terms; t++) {
    if (pos_start) pos_start[t] = at;
    memcpy(out + at, enc[t].bytes.data(), enc[t].bytes.size());
    at += enc[t].bytes.size();
    if (pos_end) pos_end[t] = at;
  }
  return SB200_OK;
}

}  // extern "C"
