// bm25.cu -- hot path 2: BM25 posting-list scoring + top-k on the device (see stract_b200_bm25.h).
//
// Data layout in HBM (per segment/field)
//   postings   the tantivy postings file, byte for byte                       ~1.0-1.5 B / posting
//   fieldnorm  1 byte per doc (FieldNormReader)                               1 B / doc
//   directory  built once from the skip lists: per 128-doc block {last_doc u32, byte offset u32,
//              bit widths u16}; per term {data offset, end offset, doc_freq, first block slot}
//   signals    optional row-major [max_doc][n_cols] f64 numeric signal scores (one 32-B sector per doc at 4 cols)
//
// Kernel k_topk<MODE>: one CTA (128 threads) per query, exhaustive scoring, exact top-k.
//   The CTA walks all query terms' posting lists block-synchronously: every term keeps one decoded 128-doc
//   block in shared memory (BitPacker4x unpack: thread k extracts value k from its lane stream, block-wide
//   prefix sum of the strict deltas).  Each round takes `bound` = the smallest last-doc among the current
//   blocks; every posting with doc <= bound is final (no later block of any term can contain such a doc),
//   so membership of a doc in the other terms is a 7-step binary search in their current block.  The term
//   with the lowest slot that contains the doc "owns" it and computes the score in the reference's f32/f64
//   operation order; no sort or merge of the lists is needed.  Candidates are pushed (smem atomics) into a
//   2k-entry buffer with a running threshold exactly like TopNComputer (top_score_collector.rs:501-554);
//   when it fills, a bitonic sort keeps the best k.  Keys are (order-preserving score bits, ~doc) so the
//   result order is the reference's (score desc, doc asc) total order.
// Roofline: HBM by bytes (posting bytes + 1 B fieldnorm (+ 8 B x n_cols signals) per scored doc), but at the
// configured sizes the postings file is L2-resident and the kernel is bound by unpack/search issue rate.
#include "common.cuh"
#include "../../include/stract_b200_bm25.h"

#ifndef SB200_EMU
#include <cub/cub.cuh>
#endif
#include <algorithm>
#include <cstdlib>
#include <vector>

namespace sb200 {
uint32_t fieldnorm_value(uint8_t id);
struct MergeJob { uint32_t first_slot, n_slots, out_slot, _pad; };
}

struct sb200_signals {
  int device = 0;
  uint32_t n_cols = 0, max_doc = 0;
  sb200::DevBuf<double> rows;
};

struct sb200_segment {
  int device = 0, record = 1, stride = 8;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr;
  uint32_t max_doc = 0, n_terms = 0;
  uint64_t postings_len = 0, n_blocks = 0, n_postings = 0;
  double stage_ms = 0;
  sb200::DevBuf<uint8_t> postings, fieldnorm;
  sb200::DevBuf<uint64_t> t_data_off, t_end_off;
  sb200::DevBuf<uint32_t> t_df, t_first;
  sb200::DevBuf<uint32_t> b_last, b_off;
  sb200::DevBuf<uint16_t> b_bits, b_bw;   // b_bw: the block-wand (fieldnorm id | tf << 8) pair of every skip entry
  std::vector<uint32_t> h_df;  // host copy (query planning: Intersection sorts by size_hint)
  // per-batch scratch (grown on demand)
  sb200::DevBuf<uint32_t> q_terms, q_nterms, o_docs, o_n, q_orig;
  sb200::DevBuf<float> q_weights, q_cache, o_scores;
  sb200::DevBuf<double> o_totals, q_coeffs;
  sb200::DevBuf<unsigned long long> counters;
  // 16-byte aligned copy of every term's block region (blocks are multiples of 16 bytes) for LDG.128 unpacking
  sb200::DevBuf<uint4> a_post;
  sb200::DevBuf<uint64_t> t_aoff;           // per term, in uint4 units
  sb200::DevBuf<uint64_t> g_khi;            // per-query candidate buffers of the warp kernel
  sb200::DevBuf<uint32_t> g_klo;
  sb200::DevBuf<uint32_t> q_items;          // item -> (query slot, lo, hi, output slot), SoA
  sb200::DevBuf<sb200::MergeJob> q_jobs;
  // scratch of the unit-based AND path (bm25_and3.cuh)
  sb200::DevBuf<uint4> a3_units;            // AUnit records
  sb200::DevBuf<uint64_t> a3_off;           // per query slot: start of its candidate list
  sb200::DevBuf<uint32_t> a3_cnt, a3_key, a3_doc;
  // scratch of the multi-field signal path (bm25_multi.cuh); lives in the FIRST field's handle
  sb200::DevBuf<uint8_t> m_fields, m_ops, m_slot_field;
  sb200::DevBuf<float> m_idf_f;
  sb200::DevBuf<double> m_boost;
  // sparse result tables go to the host packed (copy_out_tables)
  sb200::DevBuf<uint32_t> p_docs, p_scores; sb200::DevBuf<uint64_t> p_off;
  uint32_t* h_pack = nullptr; size_t h_pack_words = 0;   // page-locked staging: [n counts | offsets (u64) | docs | scores]
  // positions (sb200_segment_attach_positions, bm25_phrase.cuh)
  bool has_positions = false;
  sb200::DevBuf<uint8_t> pos_file, pb_bits;
  sb200::DevBuf<uint64_t> b_pos, pt_total, pt_afirst, pt_tail, pb_off;
  sb200::DevBuf<uint32_t> pt_nb, ptail;
  sb200::DevBuf<uint4> pa;
  // scratch of the phrase path
  sb200::DevBuf<uint32_t> ph_plan, ph_cq, ph_cdoc, ph_cord;
  sb200::DevBuf<float> ph_w;
  sb200::DevBuf<unsigned long long> ph_n;
};

namespace sb200 {

constexpr int NT = 128;            // threads per CTA == postings per block
constexpr int MAXT = SB200_MAX_QUERY_TERMS;
constexpr uint32_t TERMINATED = 0x7FFFFFFFu;

struct SegView {
  const uint32_t* p32; uint64_t postings_len;
  const uint8_t* fieldnorm; uint32_t max_doc;
  const uint64_t *t_data_off, *t_end_off; const uint32_t *t_df, *t_first;
  const uint32_t *b_last, *b_off; const uint16_t* b_bits;
  int record;
};

// ------------------------------------------------------------------ directory build -------------
// one warp per term: parse [VInt skip_len] and turn the skip entries into randomly addressable block records
__global__ void k_build_directory(const uint8_t* __restrict__ postings, const sb200_term_info* __restrict__ terms,
                                  uint32_t n_terms, int stride, const uint32_t* __restrict__ t_first,
                                  uint64_t* t_data_off, uint64_t* t_end_off, uint32_t* t_df, uint32_t* b_last,
                                  uint32_t* b_off, uint16_t* b_bits, uint16_t* b_bw, uint64_t postings_len, int* err) {
  const uint32_t t = (blockIdx.x * (uint32_t)blockDim.x + threadIdx.x) >> 5;
  if (t >= n_terms) return;
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t off = terms[t].postings_off, len = terms[t].postings_len;
  const uint32_t df = terms[t].doc_freq;
  const uint32_t nfull = df >> 7, first = t_first[t];
  if (off + len > postings_len) { if (lane == 0) *err = 1; return; }
  uint64_t skip_start = off, skip_len = 0;
  if (df >= 128) {  // split_into_skips_and_postings, block_segment_postings.rs:78-88
    // every read stays inside [off, off + len): the TermInfo is caller data and may be corrupt
    int sh = 0; uint64_t p = off; bool closed = false;
    for (int i = 0; i < 10 && p < off + len; i++) { const uint8_t b = postings[p++]; skip_len |= (uint64_t)(b & 127u) << sh; if (b & 128u) { closed = true; break; } sh += 7; }
    skip_start = p;
    if (!closed || skip_len != (uint64_t)nfull * stride || skip_start + skip_len > off + len) { if (lane == 0) *err = 2; return; }
  }
  const uint64_t data_off = skip_start + skip_len;
  if (lane == 0) { t_data_off[t] = data_off; t_end_off[t] = off + len; t_df[t] = df; }
  uint32_t run = 0;
  for (uint32_t base = 0; base < nfull; base += 32) {
    const uint32_t j = base + lane;
    uint32_t size = 0, last = 0; uint16_t bits = 0, bw = 0;
    if (j < nfull) {
      const uint8_t* e = postings + skip_start + (uint64_t)j * stride;  // skip.rs:186-238
      last = (uint32_t)e[0] | ((uint32_t)e[1] << 8) | ((uint32_t)e[2] << 16) | ((uint32_t)e[3] << 24);
      const uint32_t db = e[4] & 0x3fu, strict = (e[4] >> 6) & 1u;
      const uint32_t tb = (stride >= 8) ? e[5] : 0u;
      bits = (uint16_t)(db | (strict << 6) | (tb << 8));
      size = (db + tb) * 16u;
      if (stride >= 8) { const int o = stride == 12 ? 10 : 6; bw = (uint16_t)(e[o] | ((uint32_t)e[o + 1] << 8)); }   // skip.rs:203-232
      if (db > 32 || tb > 32) *err = 3;
    }
    uint32_t incl = size;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
    if (j < nfull) { b_last[first + j] = last; b_bits[first + j] = bits; b_bw[first + j] = bw; b_off[first + j] = run + incl - size; }
    run += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) {
    b_off[first + nfull] = run; b_last[first + nfull] = TERMINATED; b_bits[first + nfull] = 0; b_bw[first + nfull] = 0;
    if (data_off + run > off + len) *err = 4;
  }
}

// ------------------------------------------------------------------ device helpers ---------------
__device__ __forceinline__ uint32_t ord_f32(float f) { const uint32_t b = __float_as_uint(f); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); }
__device__ __forceinline__ float unord_f32(uint32_t o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o); }
__device__ __forceinline__ uint64_t ord_f64(double f) { const uint64_t b = (uint64_t)__double_as_longlong(f); return (b >> 63) ? ~b : (b | 0x8000000000000000ull); }
__device__ __forceinline__ double unord_f64(uint64_t o) { return __longlong_as_double((long long)((o >> 63) ? (o & 0x7FFFFFFFFFFFFFFFull) : ~o)); }

struct TermState {
  uint64_t data_off, end_off;
  uint32_t first, nfull, df, cur_blk, len, pos, last_doc, prev_last, done, tail_done;
  float weight;
};

struct Smem {
  uint32_t* docs; uint32_t* tfs;    // [MAXT][128]
  uint32_t* stage;                   // 336 words: one packed block (<= 1024 B) or the vint tail (<= 1280 B)
  uint32_t* vals;                    // 256 tail values
  float* cache;                      // 256
  TermState* st;                     // [MAXT]
  uint64_t* khi; uint32_t* klo;      // [CAP]
  uint32_t* misc;                    // [32] scratch: warp totals, counters
};

__device__ __forceinline__ uint32_t extract_bits(const uint32_t* words, uint32_t nb, uint32_t k) {
  if (nb == 0) return 0;
  const uint32_t lane4 = k & 3u, slot = k >> 2, bit = slot * nb, w = bit >> 5, sh = bit & 31u;
  const uint32_t lo = words[w * 4 + lane4];
  const uint32_t hi = (sh + nb > 32) ? words[(w + 1) * 4 + lane4] : 0u;
  const uint32_t v = __funnelshift_r(lo, hi, sh);
  return nb == 32 ? v : (v & ((1u << nb) - 1u));
}

// inclusive scan over the 128 threads of the CTA (wrapping u32); uses misc[0..3]; two barriers
__device__ __forceinline__ uint32_t cta_scan_incl(uint32_t x, uint32_t* misc) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) { const uint32_t n = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += n; }
  if (lane == 31) misc[warp] = x;
  __syncthreads();
  uint32_t add = 0;
  for (uint32_t w = 0; w < warp; w++) add += misc[w];
  __syncthreads();
  return x + add;
}

// stage `nbytes` of the postings file starting at absolute byte `gbyte` into aligned shared words
__device__ __forceinline__ void stage_bytes(const SegView& S, uint64_t gbyte, uint32_t nbytes, uint32_t* stage) {
  const uint64_t w0 = gbyte >> 2; const uint32_t sh = (uint32_t)(gbyte & 3u) * 8u;
  const uint32_t nwords = (nbytes + 3) >> 2;
  for (uint32_t w = threadIdx.x; w < nwords; w += NT) {
    const uint32_t lo = __ldg(S.p32 + w0 + w), hi = __ldg(S.p32 + w0 + w + 1);
    stage[w] = __funnelshift_r(lo, hi, sh);
  }
}

// decode the next block of term slot s into docs[s]/tfs[s]; every thread of the CTA calls it
__device__ void decode_next(const SegView& S, Smem& M, int s) {
  TermState& T = M.st[s];
  uint32_t* docs = M.docs + s * 128; uint32_t* tfs = M.tfs + s * 128;
  __syncthreads();
  const uint32_t blk = T.cur_blk, prev_last = T.prev_last;
  if (blk < T.nfull) {
    const uint32_t idx = T.first + blk;
    const uint32_t bits = S.b_bits[idx], db = bits & 0x3fu, strict = (bits >> 6) & 1u, tb = bits >> 8;
    stage_bytes(S, T.data_off + S.b_off[idx], (db + tb) * 16u, M.stage);
    __syncthreads();
    const uint32_t k = threadIdx.x;
    const uint32_t delta = extract_bits(M.stage, db, k) + strict;
    const uint32_t tf = (S.record >= 1) ? extract_bits(M.stage + db * 4, tb, k) + strict : 1u;
    const uint32_t pre = cta_scan_incl(delta, M.misc);
    const uint32_t base = (strict && prev_last == 0) ? 0xFFFFFFFFu : prev_last;  // offset 0 == None (compression/mod.rs:36)
    docs[k] = base + pre; tfs[k] = tf;
    __syncthreads();
    if (threadIdx.x == 0) { T.len = 128; T.pos = 0; T.last_doc = docs[127]; T.prev_last = docs[127]; T.cur_blk = blk + 1; }
  } else {
    const uint32_t n = T.df - T.nfull * 128u;
    const uint64_t tail_off = T.data_off + S.b_off[T.first + T.nfull];
    const uint32_t nbytes = (uint32_t)min((uint64_t)1340, T.end_off - tail_off);
    stage_bytes(S, tail_off, nbytes, M.stage);
    for (uint32_t i = threadIdx.x; i < 256; i += NT) M.vals[i] = (i < 128) ? 0u : 1u;
    __syncthreads();
    if (threadIdx.x < 32) {  // warp 0: vint values = runs of bytes ending with the stop bit (compression/vint.rs)
      const uint8_t* bytes = (const uint8_t*)M.stage;
      const uint32_t lane = threadIdx.x;
      uint32_t seen = 0;
      const uint32_t want = (S.record >= 1) ? 2 * n : n;
      for (uint32_t base = 0; base < nbytes && seen < want; base += 32) {
        const uint32_t b = base + lane;
        const bool stop = (b < nbytes) && (bytes[b] & 0x80u);
        const unsigned m = __ballot_sync(0xffffffffu, stop);
        if (stop) {
          const uint32_t idx = seen + __popc(m & ((1u << lane) - 1u));
          if (idx < want) {
            uint32_t start = b;
            while (start > 0 && !(bytes[start - 1] & 0x80u) && b - start < 4) start--;
            uint32_t v = 0;
            for (uint32_t i = start; i <= b; i++) v += (uint32_t)(bytes[i] & 0x7Fu) << (7 * (i - start));
            M.vals[idx < n ? idx : 128 + (idx - n)] = v;
          }
        }
        seen += __popc(m);
      }
    }
    __syncthreads();
    const uint32_t k = threadIdx.x;
    const uint32_t pre = cta_scan_incl(k < n ? M.vals[k] : 0u, M.misc);
    docs[k] = (k < n) ? prev_last + pre : TERMINATED;
    tfs[k] = (k < n) ? M.vals[128 + k] : 0u;
    __syncthreads();
    if (threadIdx.x == 0) { T.len = n; T.pos = 0; T.last_doc = n ? docs[n - 1] : 0; T.prev_last = T.last_doc; T.cur_blk = blk + 1; T.tail_done = 1; }
  }
  __syncthreads();
}

// advance term slot s to the first full block (>= its cursor) whose last doc is >= L; all threads call it
__device__ void dir_skip(const SegView& S, Smem& M, int s, uint32_t L) {
  __syncthreads();
  const TermState& t = M.st[s];
  const uint32_t first = t.first, nfull = t.nfull, tid = threadIdx.x;
  uint32_t j = nfull;
  for (uint32_t base = t.cur_blk; base < nfull; base += NT) {
    const uint32_t idx = base + tid;
    const bool pred = idx < nfull && __ldg(S.b_last + first + idx) >= L;
    const unsigned m = __ballot_sync(0xffffffffu, pred);
    if ((tid & 31) == 0) M.misc[tid >> 5] = m ? base + (tid & ~31u) + (uint32_t)__ffs(m) - 1u : 0xFFFFFFFFu;
    __syncthreads();
    const uint32_t best = min(min(M.misc[0], M.misc[1]), min(M.misc[2], M.misc[3]));
    __syncthreads();
    if (best != 0xFFFFFFFFu) { j = best; break; }
  }
  if (tid == 0) {
    TermState& w = M.st[s];
    if (j > w.cur_blk) { w.cur_blk = j; w.prev_last = S.b_last[first + j - 1]; }
  }
  __syncthreads();
}

// first index in the sorted 128-entry block with value >= x (branchless, block_search.rs:23-34)
__device__ __forceinline__ uint32_t lower_bound128(const uint32_t* a, uint32_t x) {
  uint32_t start = 0;
#pragma unroll
  for (uint32_t len = 64; len >= 1; len >>= 1) if (a[start + len - 1] < x) start += len;
  // the 7 halving steps count at most 127 smaller elements (the reference may assume target <= last element,
  // we may not): one more probe makes the result 128 when every element is smaller
  if (a[start] < x) start++;
  return start;
}

__device__ __forceinline__ bool key_gt(uint64_t ah, uint32_t al, uint64_t bh, uint32_t bl) { return ah > bh || (ah == bh && al > bl); }

// sort the CAP-entry key buffer descending (bitonic), CAP a power of two
__device__ void sort_keys_desc(Smem& M, uint32_t cap) {
  for (uint32_t size = 2; size <= cap; size <<= 1) {
    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (uint32_t i = threadIdx.x; i < (cap >> 1); i += NT) {
        const uint32_t lo = 2 * i - (i & (stride - 1));
        const uint32_t hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const uint64_t ah = M.khi[lo], bh = M.khi[hi]; const uint32_t al = M.klo[lo], bl = M.klo[hi];
        const bool swap = desc ? key_gt(bh, bl, ah, al) : key_gt(ah, al, bh, bl);
        if (swap) { M.khi[lo] = bh; M.klo[lo] = bl; M.khi[hi] = ah; M.klo[hi] = al; }
      }
    }
  }
  __syncthreads();
}

struct Params {
  SegView S;
  const uint32_t* q_terms; const uint32_t* q_nterms; const float* q_weights; const float* cache;
  const uint32_t* q_orig;   // slot -> caller's query index (slots are ordered by decreasing work)
  uint32_t n_terms_max, k, cap;
  // path B
  float k1p1; double coeff_text; const double* sig; uint32_t n_cols; const double* coeffs; uint32_t max_docs;
  // out
  uint32_t* o_docs; float* o_scores; double* o_totals; uint32_t* o_n; unsigned long long* counters;
};

// MODE 0: AND (tantivy Intersection order), 1: OR (tantivy weights, query-order sum), 2: Stract signal combine
template <int MODE>
__global__ void __launch_bounds__(NT) k_topk(const Params P) {
  SB_DYN_SMEM(smem_raw);
  Smem M;
  {
    unsigned char* p = smem_raw;
    M.khi = (uint64_t*)p; p += (size_t)P.cap * 8;
    M.st = (TermState*)p; p += sizeof(TermState) * MAXT;
    M.klo = (uint32_t*)p; p += (size_t)P.cap * 4;
    M.docs = (uint32_t*)p; p += MAXT * 128 * 4;
    M.tfs = (uint32_t*)p; p += MAXT * 128 * 4;
    M.stage = (uint32_t*)p; p += 344 * 4;
    M.vals = (uint32_t*)p; p += 256 * 4;
    M.cache = (float*)p; p += 256 * 4;
    M.misc = (uint32_t*)p;
  }
  const SegView& S = P.S;
  const uint32_t q = blockIdx.x;
  const uint32_t oq = P.q_orig ? P.q_orig[q] : q;
  const uint32_t T = P.q_nterms[q];
  const uint32_t tid = threadIdx.x;
  uint32_t* s_count = M.misc + 8;     // entries in the key buffer
  uint32_t* s_flag = M.misc + 9;      // threshold valid
  uint32_t* s_rstart = M.misc + 12;   // [MAXT+1] prefix of the round's per-term entry counts
  uint32_t* s_rhi = M.misc + 22;      // [MAXT]
  uint64_t* s_thr_hi = (uint64_t*)(M.misc + 30); uint32_t* s_thr_lo = M.misc + 10;
  for (uint32_t i = tid; i < 256; i += NT) M.cache[i] = P.cache[i];
  for (uint32_t i = tid; i < P.cap; i += NT) { M.khi[i] = 0; M.klo[i] = 0; }
  if (tid < MAXT) {
    TermState& t = M.st[tid];
    t.done = 1; t.len = 0; t.pos = 0;
    if (tid < T) {
      const uint32_t ord = P.q_terms[(size_t)q * P.n_terms_max + tid];
      t.data_off = S.t_data_off[ord]; t.end_off = S.t_end_off[ord]; t.first = S.t_first[ord]; t.df = S.t_df[ord];
      t.nfull = t.df >> 7; t.cur_blk = 0; t.last_doc = 0; t.prev_last = 0; t.tail_done = 0;
      t.done = (t.df == 0); t.weight = P.q_weights[(size_t)q * P.n_terms_max + tid];
    }
  }
  if (tid == 0) { *s_count = 0; *s_flag = 0; *s_thr_hi = 0; *s_thr_lo = 0; }
  __syncthreads();
  unsigned long long my_docs = 0, my_blocks = 0;
  unsigned bad_doc = 0u;
  uint32_t cand_seen = 0;  // path B short-circuit counter (uniform)
  bool stop_all = (T == 0);
  // watchdog: every pass of the loop below consumes a block, skips blocks or advances a cursor; a corrupt file
  // must not be able to spin a CTA forever
  unsigned long long budget = 64;
  for (uint32_t s = 0; s < T; s++) budget += 132ull * (M.st[s].nfull + 2);

  while (!stop_all) {
    if (budget-- == 0) { if (tid == 0) atomicAdd(P.counters + 2, 1ull); break; }
    // (1) refill exhausted blocks.  AND: a match is >= every term's head, so before decoding the next block of a
    // term we jump over every block whose last doc is below L = max head of the other terms, using the block
    // directory (the skip-list seek of Intersection::advance, intersection.rs:95-125 / skip.rs:243-254).
    for (uint32_t s = 0; s < T; s++) {
      const TermState& t = M.st[s];
      if (!t.done && t.pos >= t.len) {
        if (MODE == 0 && T > 1) {
          uint32_t L = 0;
          for (uint32_t x = 0; x < T; x++) { const TermState& u = M.st[x]; if (x != s && !u.done && u.pos < u.len) L = max(L, M.docs[x * 128 + u.pos]); }
          if (L > 0 && t.cur_blk < t.nfull) dir_skip(S, M, s, L);
        }
        const bool more = (t.cur_blk < t.nfull) || (t.cur_blk == t.nfull && !t.tail_done && (t.df & 127u));
        if (more) { decode_next(S, M, s); my_blocks++; }
        else { __syncthreads(); if (tid == 0) M.st[s].done = 1; __syncthreads(); }
      }
    }
    // (1b) AND: blocks already decoded but entirely below L are dead, and so are the leading docs below L
    if (MODE == 0 && T > 1) {
      bool alive = true; uint32_t L = 0;
      for (uint32_t s = 0; s < T; s++) { const TermState& t = M.st[s]; if (t.done) alive = false; else L = max(L, M.docs[s * 128 + t.pos]); }
      if (alive) {
        bool dead = false;
        for (uint32_t s = 0; s < T; s++) if (M.st[s].last_doc < L) dead = true;
        __syncthreads();
        if (tid < T) {
          TermState& w = M.st[tid];
          if (w.last_doc < L) { w.pos = 0; w.len = 0; }  // refill (with directory skip) next pass
          else { const uint32_t p = lower_bound128(M.docs + tid * 128, L); if (p > w.pos) w.pos = min(p, w.len); }
        }
        __syncthreads();
        if (dead) continue;
      }
    }
    // (2) the round's bound
    uint32_t bound = 0xFFFFFFFFu; bool any = false, all = true;
    for (uint32_t s = 0; s < T; s++) { const TermState& t = M.st[s]; if (!t.done) { bound = min(bound, t.last_doc); any = true; } else all = false; }
    if (!any || (MODE == 0 && !all)) break;
    // (3) per-term ranges [pos, hi): docs <= bound
    if (tid < T) {
      const TermState& t = M.st[tid];
      uint32_t hi = t.pos;
      if (!t.done) { hi = lower_bound128(M.docs + tid * 128, bound + 1u); if (hi > t.len) hi = t.len; if (bound == 0xFFFFFFFFu) hi = t.len; }
      s_rhi[tid] = hi;
    }
    __syncthreads();
    if (tid == 0) {
      uint32_t acc = 0;
      for (uint32_t s = 0; s < T; s++) { s_rstart[s] = acc; if (MODE != 0 || s == 0) acc += s_rhi[s] - M.st[s].pos; }
      s_rstart[T] = acc;
    }
    __syncthreads();
    const uint32_t R = s_rstart[T];
    if (*s_count + R > P.cap) {  // make room: keep the best k (TopNComputer::truncate_top_n)
      sort_keys_desc(M, P.cap);
      if (tid == 0) {
        const uint32_t c = min(*s_count, P.k);
        *s_count = c;
        if (c == P.k) { *s_flag = 1; *s_thr_hi = M.khi[P.k - 1]; *s_thr_lo = M.klo[P.k - 1]; }
      }
      __syncthreads();
      for (uint32_t i = P.k + tid; i < P.cap; i += NT) { M.khi[i] = 0; M.klo[i] = 0; }
      __syncthreads();
    }
    uint32_t cutoff = 0xFFFFFFFFu;  // path B short circuit: largest doc still inside max_docs
    bool last_round = false;
    if (MODE == 2 && P.max_docs) {
      // count this round's owners; if they overflow max_docs, find the doc cutoff by sorting them
      uint32_t mine = 0;
      for (uint32_t e = tid; e < R; e += NT) {
        uint32_t i = 0; while (e >= s_rstart[i + 1]) i++;
        const uint32_t d = M.docs[i * 128 + M.st[i].pos + (e - s_rstart[i])];
        bool owner = true;
        for (uint32_t x = 0; x < i && owner; x++) if (!M.st[x].done) { const uint32_t j = lower_bound128(M.docs + x * 128, d); if (j < M.st[x].len && M.docs[x * 128 + j] == d) owner = false; }
        mine += owner;
      }
      const uint32_t incl = cta_scan_incl(mine, M.misc);
      const uint32_t round_owners = __shfl_sync(0xffffffffu, incl, 31);  // lane 31 of the last warp has the total...
      __syncthreads();
      if (tid == NT - 1) M.misc[4] = incl;
      __syncthreads();
      const uint32_t total_owners = M.misc[4]; (void)round_owners;
      if (cand_seen + total_owners >= P.max_docs) {
        last_round = true;
        const uint32_t remaining = P.max_docs - cand_seen;
        // owners' docs -> vals/stage scratch is too small for 1024; reuse the (sorted, truncated) tail of the key buffer?  simpler:
        // select the `remaining`-th smallest owner doc by counting: binary search on the doc value
        uint32_t lo = 0, hi = bound;
        while (lo < hi) {
          const uint32_t mid = lo + ((hi - lo) >> 1);
          uint32_t c = 0;
          for (uint32_t e = tid; e < R; e += NT) {
            uint32_t i = 0; while (e >= s_rstart[i + 1]) i++;
            const uint32_t d = M.docs[i * 128 + M.st[i].pos + (e - s_rstart[i])];
            if (d > mid) continue;
            bool owner = true;
            for (uint32_t x = 0; x < i && owner; x++) if (!M.st[x].done) { const uint32_t j = lower_bound128(M.docs + x * 128, d); if (j < M.st[x].len && M.docs[x * 128 + j] == d) owner = false; }
            c += owner;
          }
          const uint32_t inc2 = cta_scan_incl(c, M.misc);
          __syncthreads();
          if (tid == NT - 1) M.misc[4] = inc2;
          __syncthreads();
          if (M.misc[4] >= remaining) hi = mid; else lo = mid + 1;
          __syncthreads();
        }
        cutoff = lo;
      }
      cand_seen += total_owners;
    }
    // (4) score the round's postings
    const bool thr_on = *s_flag != 0; const uint64_t thr_hi = *s_thr_hi; const uint32_t thr_lo = *s_thr_lo;
    for (uint32_t e = tid; e < R; e += NT) {
      uint32_t i = 0; while (e >= s_rstart[i + 1]) i++;
      const uint32_t j = M.st[i].pos + (e - s_rstart[i]);
      const uint32_t d = M.docs[i * 128 + j];
      if (d > cutoff) continue;
      uint32_t tf[MAXT];
      bool ok = true;
#pragma unroll
      for (uint32_t x = 0; x < MAXT; x++) {
        tf[x] = 0;
        if (x >= T || !ok) continue;
        if (x == i) { tf[x] = M.tfs[i * 128 + j]; continue; }
        bool found = false;
        if (!M.st[x].done) {
          const uint32_t jj = lower_bound128(M.docs + x * 128, d);
          if (jj < M.st[x].len && M.docs[x * 128 + jj] == d) { found = true; tf[x] = M.tfs[x * 128 + jj]; }
        }
        if (MODE == 0) { if (!found) ok = false; }
        else if (found && x < i) ok = false;  // a lower slot owns this doc
      }
      if (!ok) continue;
      if (d >= S.max_doc) { bad_doc = 1u; continue; }  // corrupt deltas: never index the doc tables with it
      my_docs++;
      const uint32_t fid = S.fieldnorm[d];
      const float norm = M.cache[fid];
      uint64_t khi;
      if (MODE == 2) {
        float bm = 0.0f;  // MultiBm25Weight::score: f32 sum over the query terms in query order (bm25.rs:97-102)
#pragma unroll
        for (uint32_t x = 0; x < MAXT; x++) if (x < T) {
          float sc = 0.0f;
          if (tf[x]) { const float t = (float)tf[x]; sc = __fmul_rn(M.st[x].weight, __fdiv_rn(__fmul_rn(t, P.k1p1), __fadd_rn(t, norm))); }
          bm = __fadd_rn(bm, sc);
        }
        double total = __dadd_rn(0.0, __dmul_rn(P.coeff_text, (double)bm));  // initial.rs:80-85: sum of coefficient * score
        for (uint32_t c = 0; c < P.n_cols; c++) total = __dadd_rn(total, __dmul_rn(P.coeffs[c], P.sig[(size_t)d * P.n_cols + c]));
        khi = ord_f64(total);
      } else {
        float sc[MAXT];
#pragma unroll
        for (uint32_t x = 0; x < MAXT; x++) { sc[x] = 0.0f; if (x < T && tf[x]) { const float t = (float)tf[x]; sc[x] = __fmul_rn(M.st[x].weight, __fdiv_rn(t, __fadd_rn(t, norm))); } }
        float total;
        if (MODE == 0) {  // Intersection::score = left + right + sum(others) (intersection.rs:153-157)
          if (T == 1) total = sc[0];
          else {
            float others = 0.0f;
#pragma unroll
            for (uint32_t x = 2; x < MAXT; x++) if (x < T) others = __fadd_rn(others, sc[x]);
            total = __fadd_rn(__fadd_rn(sc[0], sc[1]), others);
          }
        } else {
          total = 0.0f;
#pragma unroll
          for (uint32_t x = 0; x < MAXT; x++) if (x < T && tf[x]) total = __fadd_rn(total, sc[x]);
        }
        khi = (uint64_t)ord_f32(total) << 32;
      }
      const uint32_t klo = ~d;
      if (thr_on && !key_gt(khi, klo, thr_hi, thr_lo)) continue;
      const uint32_t at = atomicAdd(s_count, 1u);
      M.khi[at] = khi; M.klo[at] = klo;
    }
    __syncthreads();
    if (tid < T && !M.st[tid].done && (MODE != 0 || true)) M.st[tid].pos = s_rhi[tid];
    __syncthreads();
    if (last_round) break;
  }
  // final: sort and emit the best k
  sort_keys_desc(M, P.cap);
  const uint32_t n = min(*s_count, P.k);
  for (uint32_t i = tid; i < n; i += NT) {
    P.o_docs[(size_t)oq * P.k + i] = ~M.klo[i];
    if (MODE == 2) P.o_totals[(size_t)oq * P.k + i] = unord_f64(M.khi[i]);
    else P.o_scores[(size_t)oq * P.k + i] = unord_f32((uint32_t)(M.khi[i] >> 32));
  }
  if (tid == 0) P.o_n[oq] = n;
  if (bad_doc) atomicAdd(P.counters + 2, 1ull);  // a decoded doc id outside the segment: reported like a decode failure
  for (int o = 16; o; o >>= 1) { my_docs += __shfl_down_sync(0xffffffffu, my_docs, o); }
  if ((tid & 31) == 0 && my_docs) atomicAdd(P.counters + 0, my_docs);
  if (tid == 0 && my_blocks) atomicAdd(P.counters + 1, my_blocks);
}

__global__ void k_interleave_signals(const double* const* cols, uint32_t n_cols, uint32_t max_doc, double* rows) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= (uint64_t)max_doc * n_cols) return;
  const uint32_t d = (uint32_t)(i / n_cols), c = (uint32_t)(i % n_cols);
  rows[i] = cols[c][d];
}

// The numeric CoreSignals' value -> score transforms (core/src/ranking/signals/core/non_text.rs:25-101 and the per-signal
// `compute`), one thread per document, written straight into column `c` of the row-major table.  Every expression is the
// reference's f64 expression with explicitly rounded operations; score_rank (a libm `ln`) is not here -- see the host side.
__global__ void k_numeric_score(uint32_t kind, uint32_t dtype, const void* __restrict__ raw, uint32_t max_doc, double p0, double p1,
                                const double* __restrict__ lut, uint32_t lut_len, double* __restrict__ rows, uint32_t n_cols, uint32_t c) {
  const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= max_doc) return;
  unsigned long long u = 0; double f = 0.0;
  if (dtype == SB200_NUM_F64) f = ((const double*)raw)[d];
  else if (dtype == SB200_NUM_U64) { u = ((const unsigned long long*)raw)[d]; f = __ull2double_rn(u); }
  else { u = ((const uint8_t*)raw)[d] ? 1ull : 0ull; f = (double)u; }
  double s = 0.0;
  switch (kind) {
    case SB200_NUM_IDENTITY: s = f; break;                                                   // HostCentrality, PageCentrality (:117-155, :203-241)
    case SB200_NUM_BOOL: s = u ? 1.0 : 0.0; break;                                           // IsHomepage (:289-332)
    case SB200_NUM_BOOL_NOT: s = u ? 0.0 : 1.0; break;                                       // HasAds: score = !has_ads (:730-771)
    case SB200_NUM_INVERSE: s = __ddiv_rn(1.0, __dadd_rn(f, 1.0)); break;                    // score_trackers / digits / slashes (:61-74)
    case SB200_NUM_FETCH_TIME: s = u >= 1000ull ? 0.0 : __ddiv_rn(1.0, __dadd_rn(f, 1.0)); break;   // fetch_time_ms_cache (computer/mod.rs:257-259)
    case SB200_NUM_UPDATE_TIME: {                                                            // score_timestamp (:25-42) over update_time_cache
      const unsigned long long now = (unsigned long long)p0;                                 //   (computer/mod.rs:261-265), 72 / (hours + 72)
      if (u < now) {
        unsigned long long secs = now - u; if (secs < 1ull) secs = 1ull;
        const unsigned long long hours = secs / 3600ull;
        if (hours < 3ull * 365ull * 24ull) s = __ddiv_rn(72.0, __dadd_rn(__ull2double_rn(hours), 72.0));
      }
      break;
    }
    case SB200_NUM_LINK_DENSITY: s = f > 0.5 ? 0.0 : __dsub_rn(1.0, f); break;               // score_link_density (:76-83)
    case SB200_NUM_REGION: {                                                                 // score_region (:85-101): boost + count / total
      if (lut) {                                                                             //   lut absent = no RegionCount: the signal is 0
        const double boost = (p1 != 0.0 && u == (unsigned long long)p0) ? 50.0 : 0.0;         //   p1: a region other than All is selected, p0: its id
        s = __dadd_rn(boost, u < lut_len ? lut[u] : 0.0);
      }
      break;
    }
    default: break;
  }
  rows[(size_t)d * n_cols + c] = s;
}

static size_t smem_bytes(uint32_t cap) {
  return (size_t)cap * 12 + sizeof(TermState) * MAXT + MAXT * 128 * 8 + 344 * 4 + 256 * 4 + 256 * 4 + 40 * 4;
}

template <int MODE>
static int launch_topk(const Params& P, uint32_t n_queries, cudaStream_t s) {
  const size_t sm = smem_bytes(P.cap);
  static size_t configured[3] = {0, 0, 0};
  if (sm > 48 * 1024 && configured[MODE] < sm) {
    SB_CUDA(cudaFuncSetAttribute(k_topk<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    configured[MODE] = sm;
  }
  SB_LAUNCH(k_topk<MODE>, n_queries, NT, sm, s, P);
  SB_CHECK_LAUNCH();
  return SB200_OK;
}

template <class T>
static int ensure(DevBuf<T>& b, size_t n) { if (b.n < n) return b.alloc(n + (n >> 2) + 16); return SB200_OK; }

}  // namespace sb200
#include "tma.cuh"
#include "bm25_warp.cuh"
namespace sb200 {

template <int MODE>
static int launch_topk_warp(const WParams& P, cudaStream_t s) {
  const size_t per_warp = (size_t)P.n_terms_max * 128 * 8 + sizeof(WTerm) * P.n_terms_max + 32 * 4;
  const size_t sm = 1024 + WQ * per_warp;
  static size_t configured[3] = {0, 0, 0};
  if (sm > 48 * 1024 && configured[MODE] < sm) {
    SB_CUDA(cudaFuncSetAttribute(k_topk_warp<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    configured[MODE] = sm;
  }
  SB_LAUNCH(k_topk_warp<MODE>, div_up(P.n_items, WQ), WQ * 32, sm, s, P);
  SB_CHECK_LAUNCH();
  return SB200_OK;
}

}  // namespace sb200
#include "bm25_and3.cuh"
#include "bm25_or3.cuh"
#include "bm25_multi.cuh"
#include "bm25_wand.cuh"
#include "bm25_phrase.cuh"
namespace sb200 {

static void seg_view(const sb200_segment* g, SegView& S) {
  S.p32 = (const uint32_t*)g->postings.p; S.postings_len = g->postings_len; S.fieldnorm = g->fieldnorm.p; S.max_doc = g->max_doc;
  S.t_data_off = g->t_data_off.p; S.t_end_off = g->t_end_off.p; S.t_df = g->t_df.p; S.t_first = g->t_first.p;
  S.b_last = g->b_last.p; S.b_off = g->b_off.p; S.b_bits = g->b_bits.p; S.record = g->record;
}

// Work items of a batch whose query slots are ordered by decreasing work: a query much larger than the average is cut
// into <= 16 doc ranges (W*k <= 16384 for the merge); their partial top-k lists are merged by k_merge_topk.
struct ItemPlan {
  std::vector<uint32_t> q, lo, hi, out;
  std::vector<MergeJob> jobs;
  uint32_t extra = 0, capm = 0;
};
static void plan_items(const std::vector<uint64_t>& work, const std::vector<uint32_t>& order, uint32_t k, uint32_t max_doc, bool can_split, ItemPlan& pl) {
  const uint32_t nq = (uint32_t)work.size();
  uint64_t total = 0;
  for (uint64_t w : work) total += w;
  const uint64_t target = std::max<uint64_t>(32768, total / std::max<uint32_t>(nq, 1));
  const uint32_t wmax = std::max<uint32_t>(1, std::min<uint32_t>(16, 16384 / k));
  for (uint32_t slot = 0; slot < nq; slot++) {
    uint32_t W = can_split ? (uint32_t)std::min<uint64_t>(wmax, (work[slot] + target - 1) / target) : 1;
    if (W < 1) W = 1;
    if (W == 1) { pl.q.push_back(slot); pl.lo.push_back(0); pl.hi.push_back(0xFFFFFFFFu); pl.out.push_back(order[slot]); continue; }
    MergeJob j; j.first_slot = nq + pl.extra; j.n_slots = W; j.out_slot = order[slot]; j._pad = 0;
    pl.jobs.push_back(j);
    for (uint32_t c = 0; c < W; c++) {
      pl.q.push_back(slot);
      pl.lo.push_back((uint32_t)((uint64_t)max_doc * c / W));
      pl.hi.push_back(c + 1 == W ? 0xFFFFFFFFu : (uint32_t)((uint64_t)max_doc * (c + 1) / W));
      pl.out.push_back(nq + pl.extra + c);
    }
    pl.extra += W;
  }
  if (!pl.jobs.empty()) { pl.capm = 1024; while (pl.capm < wmax * k) pl.capm <<= 1; }
}

template <int TMAX>
static int launch_multi(const MParams& P, cudaStream_t s) {
  const size_t sm = m_cta_smem<TMAX>();
  static bool configured = false;
  if (!configured) { SB_CUDA(cudaFuncSetAttribute(k_sig_multi<TMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm)); configured = true; }
  SB_LAUNCH(k_sig_multi<TMAX>, div_up(P.n_items, WQ), WQ * 32, sm, s, P);
  SB_CHECK_LAUNCH();
  return SB200_OK;
}

static int run_multi(const sb200_multi_signal_batch* b, uint32_t* docs, double* totals, uint32_t* n_out, sb200_bm25_stats* stats) {
  if (!b || !b->fields || !b->ops || !b->slot_field || !b->slot_term || !b->slot_idf || !b->slot_idf_f || !docs || !totals || !n_out)
    SB_FAIL(SB200_EINVAL, "NULL argument");
  const uint32_t nq = b->n_queries, SM = b->n_slots, k = b->k, NF = b->n_fields, NO = b->n_ops;
  if (NF == 0 || NF > (uint32_t)M_MAX_FIELDS) SB_FAIL(SB200_ERANGE, "n_fields %u outside [1,%d]", NF, M_MAX_FIELDS);
  if (NO == 0 || NO > (uint32_t)M_MAX_OPS) SB_FAIL(SB200_ERANGE, "n_ops %u outside [1,%d]", NO, M_MAX_OPS);
  if (SM == 0 || SM > 16) SB_FAIL(SB200_ERANGE, "n_slots %u outside [1,16]", SM);
  if (k == 0 || k > SB200_MAX_K) SB_FAIL(SB200_ERANGE, "k %u outside [1,%d]", k, SB200_MAX_K);
  sb200_segment* g = b->fields[0].seg;
  if (!g) SB_FAIL(SB200_EINVAL, "field 0 has no segment");
  SB_CUDA(cudaSetDevice(g->device));
  cudaStream_t s = g->stream;
  for (uint32_t f = 0; f < NF; f++) {
    const sb200_segment* x = b->fields[f].seg;
    if (!x || !b->fields[f].tf_cache256) SB_FAIL(SB200_EINVAL, "field %u: NULL segment or cache", f);
    if (x->device != g->device || x->max_doc != g->max_doc) SB_FAIL(SB200_EINVAL, "field %u is not a field of the same segment (device / max_doc differ)", f);
  }
  uint32_t n_cols = 0;
  for (uint32_t o = 0; o < NO; o++) {
    const sb200_signal_op& op = b->ops[o];
    if (op.kind > 4u) SB_FAIL(SB200_EINVAL, "op %u: kind %u", o, op.kind);
    if (op.kind != 4u && op.kind != 1u && op.field >= NF) SB_FAIL(SB200_EINVAL, "op %u: field %u >= %u", o, op.field, NF);
    if (op.kind == 4u) {
      if (!b->signals || op.col >= b->signals->n_cols) SB_FAIL(SB200_EINVAL, "op %u: numeric column %u not in the signal table", o, op.col);
      n_cols = b->signals->n_cols;
    }
  }
  if (n_cols && b->signals->max_doc < g->max_doc) SB_FAIL(SB200_EINVAL, "signal table covers %u docs, segment has %u", b->signals->max_doc, g->max_doc);
  if (nq == 0) return SB200_OK;
  // planning: slots keep their query order (the f32 sums depend on it); padding slots (field 0xFF) are dropped
  std::vector<uint8_t> sf((size_t)nq * SM, 0);
  std::vector<uint32_t> st((size_t)nq * SM, SB200_NO_TERM), ns(nq, 0), order(nq);
  std::vector<float> w1((size_t)nq * SM, 0.f), w2((size_t)nq * SM, 0.f);
  std::vector<double> wb(b->slot_boost ? (size_t)nq * SM : 0, 0.0);
  std::vector<uint64_t> work(nq, 0), work_sorted(nq, 0);
  unsigned long long postings = 0;
  for (uint32_t q = 0; q < nq; q++) {
    order[q] = q;
    for (uint32_t x = 0; x < SM; x++) {
      const uint8_t f = b->slot_field[(size_t)q * SM + x];
      if (f == 0xFF) continue;
      if ((f & 0x7F) >= NF) SB_FAIL(SB200_EINVAL, "query %u slot %u: field %u >= %u", q, x, (unsigned)(f & 0x7F), NF);
      if ((f & 0x80) && !b->slot_boost) SB_FAIL(SB200_EINVAL, "query %u slot %u is a rule slot but slot_boost is NULL", q, x);
      const uint32_t ord = b->slot_term[(size_t)q * SM + x];
      if (ord != SB200_NO_TERM && ord < b->fields[f & 0x7F].seg->n_terms) work[q] += b->fields[f & 0x7F].seg->h_df[ord];
    }
    postings += work[q];
  }
  std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t c) { return work[a] > work[c]; });
  for (uint32_t slot = 0; slot < nq; slot++) {
    const uint32_t q = order[slot];
    uint32_t c = 0;
    for (int pass = 0; pass < 2; pass++)   // text slots first (query order kept), rule docsets behind them (rule order kept)
      for (uint32_t x = 0; x < SM; x++) {
        const uint8_t f = b->slot_field[(size_t)q * SM + x];
        if (f == 0xFF || ((f & 0x80) != 0) != (pass == 1)) continue;
        const size_t o = (size_t)slot * SM + c;
        sf[o] = f; st[o] = b->slot_term[(size_t)q * SM + x]; w1[o] = b->slot_idf[(size_t)q * SM + x]; w2[o] = b->slot_idf_f[(size_t)q * SM + x];
        if (b->slot_boost) wb[o] = b->slot_boost[(size_t)q * SM + x];
        c++;
      }
    ns[slot] = c; work_sorted[slot] = work[q];
  }
  ItemPlan pl;
  plan_items(work_sorted, order, k, g->max_doc, getenv("SB200_BM25_NOSPLIT") == nullptr, pl);
  const uint32_t n_items = (uint32_t)pl.q.size();
  const size_t n_slots_out = (size_t)nq + pl.extra;
  uint32_t cap = 1024; while (cap < k + SM * 128u) cap <<= 1;
  // device copies
  std::vector<MField> hf(NF);
  for (uint32_t f = 0; f < NF; f++) {
    memset(&hf[f], 0, sizeof(MField));
    const sb200_segment* x = b->fields[f].seg;
    seg_view(x, hf[f].S); hf[f].a128 = x->a_post.p; hf[f].t_aoff = x->t_aoff.p;
    memcpy(hf[f].cache, b->fields[f].tf_cache256, 256 * 4);
    hf[f].k1p1 = b->fields[f].k1 + 1.0f; hf[f].coef = b->fields[f].bm25f_coefficient; hf[f].n_terms = x->n_terms;
  }
  std::vector<MOp> ho(NO);
  for (uint32_t o = 0; o < NO; o++) { ho[o].kind = b->ops[o].kind; ho[o].field = b->ops[o].field; ho[o].chain = b->ops[o].chain; ho[o].col = b->ops[o].col; ho[o].coeff = b->ops[o].coeff; }
  SB_TRY(ensure(g->m_fields, NF * sizeof(MField))); SB_TRY(ensure(g->m_ops, NO * sizeof(MOp))); SB_TRY(ensure(g->m_slot_field, (size_t)nq * SM));
  SB_TRY(ensure(g->q_terms, (size_t)nq * SM)); SB_TRY(ensure(g->q_weights, (size_t)nq * SM)); SB_TRY(ensure(g->m_idf_f, (size_t)nq * SM));
  SB_TRY(ensure(g->q_nterms, nq)); SB_TRY(ensure(g->q_orig, nq)); SB_TRY(ensure(g->o_docs, n_slots_out * k)); SB_TRY(ensure(g->o_n, n_slots_out));
  SB_TRY(ensure(g->o_totals, n_slots_out * k)); SB_TRY(ensure(g->counters, 4));
  SB_TRY(ensure(g->q_items, (size_t)4 * n_items)); SB_TRY(ensure(g->q_jobs, pl.jobs.size() + 1));
  SB_TRY(ensure(g->g_khi, (size_t)n_items * cap)); SB_TRY(ensure(g->g_klo, (size_t)n_items * cap));
  SB_CUDA(cudaEventRecord(g->ev0, s));
  SB_CUDA(cudaMemcpyAsync(g->m_fields.p, hf.data(), NF * sizeof(MField), cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->m_ops.p, ho.data(), NO * sizeof(MOp), cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->m_slot_field.p, sf.data(), sf.size(), cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_terms.p, st.data(), st.size() * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_weights.p, w1.data(), w1.size() * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->m_idf_f.p, w2.data(), w2.size() * 4, cudaMemcpyHostToDevice, s));
  if (b->slot_boost) { SB_TRY(ensure(g->m_boost, wb.size())); SB_CUDA(cudaMemcpyAsync(g->m_boost.p, wb.data(), wb.size() * 8, cudaMemcpyHostToDevice, s)); }
  SB_CUDA(cudaMemcpyAsync(g->q_nterms.p, ns.data(), ns.size() * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_orig.p, order.data(), (size_t)nq * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_items.p, pl.q.data(), (size_t)n_items * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_items.p + n_items, pl.lo.data(), (size_t)n_items * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_items.p + 2 * (size_t)n_items, pl.hi.data(), (size_t)n_items * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_items.p + 3 * (size_t)n_items, pl.out.data(), (size_t)n_items * 4, cudaMemcpyHostToDevice, s));
  if (!pl.jobs.empty()) SB_CUDA(cudaMemcpyAsync(g->q_jobs.p, pl.jobs.data(), pl.jobs.size() * sizeof(MergeJob), cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemsetAsync(g->counters.p, 0, 4 * sizeof(unsigned long long), s));
  MParams P;
  memset(&P, 0, sizeof(P));
  P.fields = (const MField*)g->m_fields.p; P.n_fields = NF; P.max_doc = g->max_doc;
  P.ops = (const MOp*)g->m_ops.p; P.n_ops = NO;
  P.q_slot_field = g->m_slot_field.p; P.q_slot_term = g->q_terms.p; P.q_idf = g->q_weights.p; P.q_idf_f = g->m_idf_f.p; P.q_nslots = g->q_nterms.p;
  P.q_boost = b->slot_boost ? g->m_boost.p : nullptr;
  P.q_orig = g->q_orig.p; P.n_queries = nq; P.n_slots_max = SM; P.k = k; P.cap = cap;
  P.n_items = n_items; P.item_q = g->q_items.p; P.item_lo = g->q_items.p + n_items; P.item_hi = g->q_items.p + 2 * (size_t)n_items; P.item_out = g->q_items.p + 3 * (size_t)n_items;
  if (n_cols) { P.sig = b->signals->rows.p; P.n_cols = n_cols; }
  P.g_khi = g->g_khi.p; P.g_klo = g->g_klo.p; P.o_docs = g->o_docs.p; P.o_totals = g->o_totals.p; P.o_n = g->o_n.p; P.counters = g->counters.p;
  SB_CUDA(cudaEventRecord(g->evk0, s));
  if (SM <= 8) SB_TRY(launch_multi<8>(P, s)); else SB_TRY(launch_multi<16>(P, s));
  if (!pl.jobs.empty()) {
    const size_t msm = (size_t)pl.capm * 12;
    static size_t mconf = 0;
    if (msm > 48 * 1024 && mconf < msm) { SB_CUDA(cudaFuncSetAttribute(k_merge_topk<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msm)); mconf = msm; }
    SB_LAUNCH(k_merge_topk<2>, (unsigned)pl.jobs.size(), 256, msm, s, g->q_jobs.p, k, pl.capm, P.o_docs, (float*)nullptr, P.o_totals, P.o_n);
    SB_CHECK_LAUNCH();
  }
  SB_CUDA(cudaEventRecord(g->evk1, s));
  SB_CUDA(cudaMemcpyAsync(docs, g->o_docs.p, (size_t)nq * k * 4, cudaMemcpyDefault, s));
  SB_CUDA(cudaMemcpyAsync(totals, g->o_totals.p, (size_t)nq * k * 8, cudaMemcpyDefault, s));
  SB_CUDA(cudaMemcpyAsync(n_out, g->o_n.p, (size_t)nq * 4, cudaMemcpyDefault, s));
  unsigned long long h[4] = {0, 0, 0, 0};
  SB_CUDA(cudaMemcpyAsync(h, g->counters.p, sizeof(h), cudaMemcpyDeviceToHost, s));
  SB_CUDA(cudaEventRecord(g->ev1, s));
  SB_CUDA(cudaStreamSynchronize(s));
  if (h[2]) SB_FAIL(SB200_EFORMAT, "%llu queries hit the decode watchdog (inconsistent posting data)", h[2]);
  if (stats) {
    float ms = 0; cudaEventElapsedTime(&ms, g->ev0, g->ev1);
    stats->postings_scored = postings; stats->docs_scored = h[0]; stats->blocks_decoded = h[1]; stats->ms = ms; cudaEventElapsedTime(&stats->kernel_ms, g->evk0, g->evk1);
  }
  return SB200_OK;
}

// union modes through k_or3, instantiated for the smallest term-count bound that covers the batch
template <int MODE, int MINB>
static int launch_or3_occ(const WParams& P, cudaStream_t s) {
  const unsigned grid = div_up(P.n_items, WQ);
  void (*kern)(const WParams) = k_or3<MODE, 8, MINB>;
  if (P.n_terms_max <= 2) kern = k_or3<MODE, 2, MINB>;
  else if (P.n_terms_max <= 3) kern = k_or3<MODE, 3, MINB>;
  else if (P.n_terms_max <= 5) kern = k_or3<MODE, 5, MINB>;
  SB_LAUNCH(kern, grid, WQ * 32, 0, s, P);
  SB_CHECK_LAUNCH();
  return SB200_OK;
}
template <int MODE>
static int launch_or3(const WParams& P, cudaStream_t s) {
  static const int occ = [] { const char* e = getenv("SB200_OR3_OCC"); return e ? atoi(e) : 6; }();   // C5: 608 / 588 / 900 ms at 5 / 6 / 8
  if (occ >= 8) return launch_or3_occ<MODE, 8>(P, s);
  if (occ >= 6) return launch_or3_occ<MODE, 6>(P, s);
  return launch_or3_occ<MODE, 5>(P, s);
}

// Result tables to the caller.  An AND batch fills a fraction of its [n_queries][k] table (C4: 72 of 1000 entries per
// query), and the dense copy of 80 MB was a third of the end-to-end time: when the tables go to host memory and are
// less than half full, the valid prefixes are packed on the device, cross PCIe as one block and are scattered into the
// caller's tables by the host.  f32 scores only (path A); dense copy otherwise.
__global__ void k_pack_tables(const uint32_t* __restrict__ o_n, const uint64_t* __restrict__ off, const uint32_t* __restrict__ o_docs,
                              const float* __restrict__ o_scores, uint32_t k, uint32_t* p_docs, uint32_t* p_scores) {
  const uint32_t q = blockIdx.x, n = o_n[q];
  const uint64_t base = off[q];
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
    p_docs[base + i] = o_docs[(size_t)q * k + i];
    p_scores[base + i] = __float_as_uint(o_scores[(size_t)q * k + i]);
  }
}
static int copy_out_tables(sb200_segment* g, uint32_t nq, uint32_t k, uint32_t* docs, float* scores, double* totals, uint32_t* n_out) {
  cudaStream_t s = g->stream;
  const bool sparse_ok = scores && !totals && !is_device_ptr(docs) && !is_device_ptr(scores) && !is_device_ptr(n_out) &&
                         (size_t)nq * k >= (getenv("SB200_BM25_PACK_MIN") ? (size_t)atol(getenv("SB200_BM25_PACK_MIN")) : ((size_t)1 << 18)) &&
                         getenv("SB200_BM25_DENSE_OUT") == nullptr;
  if (sparse_ok) {
    const size_t head = (size_t)nq + 2 * (size_t)nq;   // counts (u32) + offsets (u64 as two words)
    if (g->h_pack_words < head) {
      if (g->h_pack) cudaFreeHost(g->h_pack);
      g->h_pack = nullptr; g->h_pack_words = 0;
      SB_CUDA(cudaMallocHost((void**)&g->h_pack, (head + 1024) * 4));
      g->h_pack_words = head + 1024;
    }
    SB_CUDA(cudaMemcpyAsync(g->h_pack, g->o_n.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaStreamSynchronize(s));
    uint64_t total = 0;
    std::vector<uint64_t> off(nq);
    for (uint32_t q = 0; q < nq; q++) { off[q] = total; total += g->h_pack[q]; }
    if (total * 2 < (uint64_t)nq * k) {
      memcpy(n_out, g->h_pack, (size_t)nq * 4);
      if (total == 0) return SB200_OK;
      SB_TRY(ensure(g->p_off, nq)); SB_TRY(ensure(g->p_docs, (size_t)total)); SB_TRY(ensure(g->p_scores, (size_t)total));
      const size_t need = head + 2 * (size_t)total;
      if (g->h_pack_words < need) {
        cudaFreeHost(g->h_pack); g->h_pack = nullptr; g->h_pack_words = 0;
        SB_CUDA(cudaMallocHost((void**)&g->h_pack, (need + (need >> 2)) * 4));
        g->h_pack_words = need + (need >> 2);
      }
      SB_CUDA(cudaMemcpyAsync(g->p_off.p, off.data(), (size_t)nq * 8, cudaMemcpyHostToDevice, s));
      SB_LAUNCH(k_pack_tables, nq, 128, 0, s, g->o_n.p, g->p_off.p, g->o_docs.p, g->o_scores.p, k, g->p_docs.p, g->p_scores.p);
      SB_CHECK_LAUNCH();
      uint32_t* hd = g->h_pack + head; uint32_t* hs = hd + total;
      SB_CUDA(cudaMemcpyAsync(hd, g->p_docs.p, (size_t)total * 4, cudaMemcpyDeviceToHost, s));
      SB_CUDA(cudaMemcpyAsync(hs, g->p_scores.p, (size_t)total * 4, cudaMemcpyDeviceToHost, s));
      SB_CUDA(cudaStreamSynchronize(s));
      for (uint32_t q = 0; q < nq; q++) {
        const uint32_t n = n_out[q];
        if (!n) continue;
        memcpy(docs + (size_t)q * k, hd + off[q], (size_t)n * 4);
        memcpy(scores + (size_t)q * k, hs + off[q], (size_t)n * 4);
      }
      return SB200_OK;
    }
    memcpy(n_out, g->h_pack, (size_t)nq * 4);
    SB_CUDA(cudaMemcpyAsync(docs, g->o_docs.p, (size_t)nq * k * 4, cudaMemcpyDefault, s));
    SB_CUDA(cudaMemcpyAsync(scores, g->o_scores.p, (size_t)nq * k * 4, cudaMemcpyDefault, s));
    return SB200_OK;
  }
  SB_CUDA(cudaMemcpyAsync(docs, g->o_docs.p, (size_t)nq * k * 4, cudaMemcpyDefault, s));
  if (totals) SB_CUDA(cudaMemcpyAsync(totals, g->o_totals.p, (size_t)nq * k * 8, cudaMemcpyDefault, s));
  else if (scores) SB_CUDA(cudaMemcpyAsync(scores, g->o_scores.p, (size_t)nq * k * 4, cudaMemcpyDefault, s));
  SB_CUDA(cudaMemcpyAsync(n_out, g->o_n.p, (size_t)nq * 4, cudaMemcpyDefault, s));
  return SB200_OK;
}

// AND batch through the unit kernel: `terms`/`nterms` are the planned clauses per query slot (sorted by doc_freq),
// results land in g->o_docs / o_scores / o_n at the caller's query index (order[slot]).  Candidate memory is
// sum(doc_freq of the rarest clause) x 8 B; slots are processed in groups that keep it under a budget.
static int run_and3(sb200_segment* g, const Params& P, const std::vector<uint32_t>& terms, const std::vector<uint32_t>& nterms,
                    uint32_t nq, uint32_t nt, uint32_t k, cudaStream_t s) {
  static_assert(sizeof(AUnit) == sizeof(uint4), "AUnit is stored in a uint4 buffer");
  uint64_t budget = (uint64_t)8 << 30;
  if (const char* e = getenv("SB200_AND3_BUDGET_MB")) { const long mb = atol(e); if (mb > 0) budget = (uint64_t)mb << 20; }
  const uint64_t max_entries = std::max<uint64_t>(budget / 8, 1);
  std::vector<uint64_t> off(nq, 0);
  std::vector<AUnit> units;
  static size_t sel_conf = 0;
  const size_t sel_smem = (size_t)A3_SEL_CAP * 8;
  if (sel_conf < sel_smem) {
    SB_CUDA(cudaFuncSetAttribute(k_and3_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sel_smem));
    sel_conf = sel_smem;
  }
  SB_TRY(ensure(g->a3_off, nq)); SB_TRY(ensure(g->a3_cnt, nq));
  uint32_t g0 = 0;
  while (g0 < nq) {
    // group [g0, g1): as many slots as fit the candidate budget (at least one)
    uint64_t entries = 0; uint32_t g1 = g0;
    units.clear();
    while (g1 < nq) {
      const uint32_t dfA = nterms[g1] ? g->h_df[terms[(size_t)g1 * nt]] : 0u;
      if (g1 > g0 && entries + dfA > max_entries) break;
      off[g1] = entries; entries += dfA;
      const uint32_t nblk = (dfA >> 7) + ((dfA & 127u) ? 1u : 0u);
      for (uint32_t b0 = 0; b0 < nblk; b0 += A3_UNIT_BLOCKS) {
        AUnit u; u.q = g1; u.blk_lo = b0; u.blk_hi = std::min(nblk, b0 + A3_UNIT_BLOCKS); u._pad = 0;
        units.push_back(u);
      }
      g1++;
    }
    const uint32_t n_units = (uint32_t)units.size();
    SB_TRY(ensure(g->a3_key, (size_t)std::max<uint64_t>(entries, 1))); SB_TRY(ensure(g->a3_doc, (size_t)std::max<uint64_t>(entries, 1)));
    SB_TRY(ensure(g->a3_units, std::max<size_t>(n_units, 1)));
    if (g0 == 0) SB_CUDA(cudaEventRecord(g->evk0, s));   // kernel_ms starts here: the unit list above is host planning
    SB_CUDA(cudaMemcpyAsync(g->a3_off.p + g0, off.data() + g0, (size_t)(g1 - g0) * 8, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemsetAsync(g->a3_cnt.p + g0, 0, (size_t)(g1 - g0) * 4, s));
    if (n_units) {
      SB_CUDA(cudaMemcpyAsync(g->a3_units.p, units.data(), (size_t)n_units * sizeof(AUnit), cudaMemcpyHostToDevice, s));
      A3Params A;
      memset(&A, 0, sizeof(A));
      A.S = P.S; A.a128 = g->a_post.p; A.t_aoff = g->t_aoff.p;
      A.q_terms = P.q_terms; A.q_nterms = P.q_nterms; A.q_weights = P.q_weights; A.cache = P.cache; A.n_terms_max = nt;
      A.units = (const AUnit*)g->a3_units.p; A.n_units = n_units;
      A.cand_off = g->a3_off.p; A.cand_cnt = g->a3_cnt.p; A.c_key = g->a3_key.p; A.c_doc = g->a3_doc.p;
      A.counters = P.counters;
      static const int occ = [] { const char* e = getenv("SB200_AND3_OCC"); return e ? atoi(e) : 8; }();   // C4: 3.66 / 3.51 / 3.09 ms at 5 / 6 / 8
      if (occ >= 8) SB_LAUNCH(k_and3<8>, div_up(n_units, A3_WARPS), A3_WARPS * 32, 0, s, A);
      else if (occ >= 6) SB_LAUNCH(k_and3<6>, div_up(n_units, A3_WARPS), A3_WARPS * 32, 0, s, A);
      else SB_LAUNCH(k_and3<5>, div_up(n_units, A3_WARPS), A3_WARPS * 32, 0, s, A);
      SB_CHECK_LAUNCH();
    }
    SB_LAUNCH(k_and3_select, g1 - g0, 256, sel_smem, s, g->a3_off.p, g->a3_cnt.p, g->a3_key.p, g->a3_doc.p, P.q_orig, g0, k,
              P.o_docs, P.o_scores, P.o_n);
    SB_CHECK_LAUNCH();
    if (g1 < nq) SB_CUDA(cudaStreamSynchronize(s));  // `units` / `off` are reused by the next group's async copies
    g0 = g1;
  }
  return SB200_OK;
}

static int run_batch(sb200_segment* g, const sb200_bm25_batch* b, int mode, const sb200_signal_batch* sb, uint32_t* docs,
                     float* scores, double* totals, uint32_t* n_out, sb200_bm25_stats* stats) {
  NvtxRange nvtx(sb ? "sb200 signal top-k batch" : "sb200 bm25 top-k batch");
  cudaStream_t s = g->stream;
  if (!b || !b->term_ords || !b->weights || !b->tf_cache256 || !docs || !n_out) SB_FAIL(SB200_EINVAL, "NULL argument");
  const uint32_t nq = b->n_queries, nt = b->n_terms, k = b->k;
  if (nt == 0 || nt > MAXT) SB_FAIL(SB200_ERANGE, "n_terms %u outside [1,%d]", nt, MAXT);
  if (k == 0 || k > SB200_MAX_K) SB_FAIL(SB200_ERANGE, "k %u outside [1,%d]", k, SB200_MAX_K);
  if (nq == 0) return SB200_OK;
  // host-side planning: drop padding; AND sorts the clauses by doc_freq (stable) like intersect_scorers (intersection.rs:24)
  std::vector<uint32_t> terms((size_t)nq * nt), nterms(nq);
  std::vector<float> weights((size_t)nq * nt);
  unsigned long long postings = 0;
  // longest-processing-time-first: one warp walks a whole query, so the batch finishes when its largest query
  // does; slots are ordered by decreasing posting count and results go back to the caller's index (q_orig)
  std::vector<uint32_t> order(nq);
  {
    std::vector<uint64_t> work(nq, 0);
    for (uint32_t q = 0; q < nq; q++) {
      order[q] = q;
      for (uint32_t t = 0; t < nt; t++) { const uint32_t ord = b->term_ords[(size_t)q * nt + t]; if (ord != SB200_NO_TERM && ord < g->n_terms) work[q] += g->h_df[ord]; }
    }
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t bb) { return work[a] > work[bb]; });
  }
  for (uint32_t slot = 0; slot < nq; slot++) {
    const uint32_t q = order[slot];
    uint32_t idx[MAXT]; uint32_t c = 0;
    for (uint32_t t = 0; t < nt; t++) {
      const uint32_t ord = b->term_ords[(size_t)q * nt + t];
      if (ord == SB200_NO_TERM) continue;
      if (ord >= g->n_terms) SB_FAIL(SB200_EINVAL, "query %u: term ordinal %u >= %u", q, ord, g->n_terms);
      idx[c++] = t;
    }
    if (mode == SB200_MODE_AND) std::stable_sort(idx, idx + c, [&](uint32_t a, uint32_t bb) { return g->h_df[b->term_ords[(size_t)q * nt + a]] < g->h_df[b->term_ords[(size_t)q * nt + bb]]; });
    for (uint32_t i = 0; i < c; i++) {
      terms[(size_t)slot * nt + i] = b->term_ords[(size_t)q * nt + idx[i]];
      weights[(size_t)slot * nt + i] = b->weights[(size_t)q * nt + idx[i]];
      postings += g->h_df[terms[(size_t)slot * nt + i]];
    }
    nterms[slot] = c;
  }
  // work items: queries much larger than the average are cut into doc ranges (<= 16, W*k <= 16384 for the merge)
  std::vector<uint32_t> it_q, it_lo, it_hi, it_out;
  std::vector<MergeJob> jobs;
  uint32_t extra = 0, capm = 0;
  {
    const bool can_split = !(sb && sb->max_docs) && !(!sb && mode == SB200_MODE_OR_WAND) && getenv("SB200_BM25_CTA") == nullptr &&
                           getenv("SB200_BM25_NOSPLIT") == nullptr;   // a replayed history cannot be cut into doc ranges
    const uint64_t target = std::max<uint64_t>(32768, postings / std::max<uint32_t>(nq, 1));
    const uint32_t wmax = std::max<uint32_t>(1, std::min<uint32_t>(16, 16384 / k));
    it_q.reserve(nq + 64); it_lo.reserve(nq + 64); it_hi.reserve(nq + 64); it_out.reserve(nq + 64);
    for (uint32_t slot = 0; slot < nq; slot++) {
      uint64_t work = 0;
      for (uint32_t i = 0; i < nterms[slot]; i++) work += g->h_df[terms[(size_t)slot * nt + i]];
      uint32_t W = can_split ? (uint32_t)std::min<uint64_t>(wmax, (work + target - 1) / target) : 1;
      if (W < 1) W = 1;
      if (W == 1) { it_q.push_back(slot); it_lo.push_back(0); it_hi.push_back(0xFFFFFFFFu); it_out.push_back(order[slot]); continue; }
      MergeJob j; j.first_slot = nq + extra; j.n_slots = W; j.out_slot = order[slot]; j._pad = 0;
      jobs.push_back(j);
      for (uint32_t c = 0; c < W; c++) {
        it_q.push_back(slot);
        it_lo.push_back((uint32_t)((uint64_t)g->max_doc * c / W));
        it_hi.push_back(c + 1 == W ? 0xFFFFFFFFu : (uint32_t)((uint64_t)g->max_doc * (c + 1) / W));
        it_out.push_back(nq + extra + c);
      }
      extra += W;
    }
    if (!jobs.empty()) { capm = 1024; while (capm < wmax * k) capm <<= 1; }
  }
  const uint32_t n_items = (uint32_t)it_q.size();
  const size_t n_slots_out = (size_t)nq + extra;
  SB_TRY(ensure(g->q_terms, (size_t)nq * nt)); SB_TRY(ensure(g->q_weights, (size_t)nq * nt)); SB_TRY(ensure(g->q_nterms, nq));
  SB_TRY(ensure(g->q_cache, 256)); SB_TRY(ensure(g->o_docs, n_slots_out * k)); SB_TRY(ensure(g->o_n, n_slots_out));
  if (totals) SB_TRY(ensure(g->o_totals, n_slots_out * k)); else SB_TRY(ensure(g->o_scores, n_slots_out * k));
  SB_TRY(ensure(g->counters, 4)); SB_TRY(ensure(g->q_orig, nq));
  SB_TRY(ensure(g->q_items, (size_t)4 * n_items)); SB_TRY(ensure(g->q_jobs, jobs.size() + 1));
  SB_CUDA(cudaEventRecord(g->ev0, s));
  SB_CUDA(cudaMemcpyAsync(g->q_orig.p, order.data(), (size_t)nq * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_items.p, it_q.data(), (size_t)n_items * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_items.p + n_items, it_lo.data(), (size_t)n_items * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_items.p + 2 * (size_t)n_items, it_hi.data(), (size_t)n_items * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_items.p + 3 * (size_t)n_items, it_out.data(), (size_t)n_items * 4, cudaMemcpyHostToDevice, s));
  if (!jobs.empty()) SB_CUDA(cudaMemcpyAsync(g->q_jobs.p, jobs.data(), jobs.size() * sizeof(MergeJob), cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_terms.p, terms.data(), terms.size() * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_weights.p, weights.data(), weights.size() * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_nterms.p, nterms.data(), nterms.size() * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(g->q_cache.p, b->tf_cache256, 256 * 4, cudaMemcpyDefault, s));
  SB_CUDA(cudaMemsetAsync(g->counters.p, 0, 4 * sizeof(unsigned long long), s));
  Params P;
  memset(&P, 0, sizeof(P));
  P.S.p32 = (const uint32_t*)g->postings.p; P.S.postings_len = g->postings_len; P.S.fieldnorm = g->fieldnorm.p; P.S.max_doc = g->max_doc;
  P.S.t_data_off = g->t_data_off.p; P.S.t_end_off = g->t_end_off.p; P.S.t_df = g->t_df.p; P.S.t_first = g->t_first.p;
  P.S.b_last = g->b_last.p; P.S.b_off = g->b_off.p; P.S.b_bits = g->b_bits.p; P.S.record = g->record;
  P.q_terms = g->q_terms.p; P.q_nterms = g->q_nterms.p; P.q_weights = g->q_weights.p; P.cache = g->q_cache.p; P.q_orig = g->q_orig.p;
  P.n_terms_max = nt; P.k = k;
  uint32_t cap = 1024; while (cap < k + nt * 128u) cap <<= 1;
  P.cap = cap;
  P.o_docs = g->o_docs.p; P.o_scores = g->o_scores.p; P.o_totals = g->o_totals.p; P.o_n = g->o_n.p; P.counters = g->counters.p;
  SB_CUDA(cudaEventRecord(g->evk0, s));
  if (sb) {
    P.k1p1 = sb->k1 + 1.0f;  // constants.k1 + 1.0 in f32 (core/src/ranking/bm25.rs:149)
    P.coeff_text = sb->coeff_text; P.max_docs = sb->max_docs;
    if (sb->signals && sb->signals->n_cols) {
      if (sb->signals->max_doc < g->max_doc) SB_FAIL(SB200_EINVAL, "signal table covers %u docs, segment has %u", sb->signals->max_doc, g->max_doc);
      if (!sb->coeffs) SB_FAIL(SB200_EINVAL, "coeffs is NULL");
      SB_TRY(ensure(g->q_coeffs, sb->signals->n_cols));
      SB_CUDA(cudaMemcpyAsync(g->q_coeffs.p, sb->coeffs, sb->signals->n_cols * 8, cudaMemcpyDefault, s));
      P.sig = sb->signals->rows.p; P.n_cols = sb->signals->n_cols; P.coeffs = g->q_coeffs.p;
    }
  }
  if (!sb && mode != SB200_MODE_AND && mode != SB200_MODE_OR && mode != SB200_MODE_OR_WAND) SB_FAIL(SB200_EINVAL, "mode %d", mode);
  if (!sb && mode == SB200_MODE_OR_WAND) {
    // block_wand replayed (bm25_wand.cuh): one warp per query slot, the reference's own pruning and summation order
    if (g->record < 1) SB_FAIL(SB200_EINVAL, "Block-WAND needs term frequencies (record option WithFreqs or above)");
    uint32_t wcap = 2; while (wcap < 2 * k) wcap <<= 1;
    SB_TRY(ensure(g->g_khi, (size_t)nq * wcap)); SB_TRY(ensure(g->g_klo, (size_t)nq * wcap));
    WandParams W;
    memset(&W, 0, sizeof(W));
    W.S = P.S; W.b_bw = g->b_bw.p; W.a128 = g->a_post.p; W.t_aoff = g->t_aoff.p;
    W.q_terms = P.q_terms; W.q_nterms = P.q_nterms; W.q_weights = P.q_weights; W.cache = P.cache; W.q_orig = P.q_orig;
    W.n_queries = nq; W.n_terms_max = nt; W.k = k; W.cap = wcap;
    W.g_khi = g->g_khi.p; W.g_klo = g->g_klo.p; W.o_docs = P.o_docs; W.o_scores = P.o_scores; W.o_n = P.o_n; W.counters = P.counters;
    SB_LAUNCH(k_wand, div_up(nq, WD_WARPS), WD_WARPS * 32, 0, s, W);
    SB_CHECK_LAUNCH();
  } else {
  const int kmode = sb ? 2 : mode;
  static const bool use_cta_kernel = getenv("SB200_BM25_CTA") != nullptr;  // the first-generation CTA-per-query kernel
  if (use_cta_kernel) {
    if (kmode == 2) SB_TRY(launch_topk<2>(P, nq, s));
    else if (kmode == 0) SB_TRY(launch_topk<0>(P, nq, s));
    else SB_TRY(launch_topk<1>(P, nq, s));
  } else if (kmode == 0 && env_flag("SB200_BM25_AND3", true) && [&] {
               // a single-clause "intersection" makes every posting a hit: its candidate list is the whole posting list and
               // the select pass would crawl through it chunk by chunk; the threshold-pruning kernel handles those batches
               for (uint32_t slot = 0; slot < nq; slot++)
                 if (nterms[slot] == 1 && g->h_df[terms[(size_t)slot * nt]] > 65536u) return false;
               return true;
             }()) {
    SB_TRY(run_and3(g, P, terms, nterms, nq, nt, k, s));  // unit-based intersection (bm25_and3.cuh); SB200_BM25_AND3=0: k_topk_warp<AND>
  } else {
    SB_TRY(ensure(g->g_khi, (size_t)n_items * cap)); SB_TRY(ensure(g->g_klo, (size_t)n_items * cap));
    WParams W;
    memset(&W, 0, sizeof(W));
    W.S = P.S; W.a128 = g->a_post.p; W.t_aoff = g->t_aoff.p;
    W.q_terms = P.q_terms; W.q_nterms = P.q_nterms; W.q_weights = P.q_weights; W.cache = P.cache; W.q_orig = P.q_orig;
    W.n_queries = nq; W.n_terms_max = nt; W.k = k; W.cap = cap;
    W.n_items = n_items; W.item_q = g->q_items.p; W.item_lo = g->q_items.p + n_items; W.item_hi = g->q_items.p + 2 * (size_t)n_items; W.item_out = g->q_items.p + 3 * (size_t)n_items;
    W.k1p1 = P.k1p1; W.coeff_text = P.coeff_text; W.sig = P.sig; W.n_cols = P.n_cols; W.coeffs = P.coeffs; W.max_docs = P.max_docs;
    W.g_khi = g->g_khi.p; W.g_klo = g->g_klo.p;
    W.o_docs = P.o_docs; W.o_scores = P.o_scores; W.o_totals = P.o_totals; W.o_n = P.o_n; W.counters = P.counters;
    W.use_tma = env_flag("SB200_BM25_TMA", true) ? 1u : 0u;
    const bool use_or3 = kmode != 0 && W.max_docs == 0 && env_flag("SB200_BM25_OR3", true);  // bm25_or3.cuh; SB200_BM25_OR3=0: k_topk_warp
    if (use_or3) { if (kmode == 2) SB_TRY(launch_or3<2>(W, s)); else SB_TRY(launch_or3<1>(W, s)); }
    else if (kmode == 2) SB_TRY(launch_topk_warp<2>(W, s));
    else if (kmode == 0) SB_TRY(launch_topk_warp<0>(W, s));
    else SB_TRY(launch_topk_warp<1>(W, s));
    if (!jobs.empty()) {
      const size_t msm = (size_t)capm * 12;
      static size_t mconf[3] = {0, 0, 0};
      if (kmode == 2) { if (msm > 48 * 1024 && mconf[2] < msm) { SB_CUDA(cudaFuncSetAttribute(k_merge_topk<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msm)); mconf[2] = msm; }
                        SB_LAUNCH(k_merge_topk<2>, (unsigned)jobs.size(), 256, msm, s, g->q_jobs.p, k, capm, P.o_docs, P.o_scores, P.o_totals, P.o_n); }
      else { if (msm > 48 * 1024 && mconf[0] < msm) { SB_CUDA(cudaFuncSetAttribute(k_merge_topk<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msm)); mconf[0] = msm; }
             SB_LAUNCH(k_merge_topk<0>, (unsigned)jobs.size(), 256, msm, s, g->q_jobs.p, k, capm, P.o_docs, P.o_scores, P.o_totals, P.o_n); }
      SB_CHECK_LAUNCH();
    }
  }
  }
  SB_CUDA(cudaEventRecord(g->evk1, s));
  SB_TRY(copy_out_tables(g, nq, k, docs, scores, totals, n_out));
  unsigned long long h[4] = {0, 0, 0, 0};
  SB_CUDA(cudaMemcpyAsync(h, g->counters.p, sizeof(h), cudaMemcpyDeviceToHost, s));
  SB_CUDA(cudaEventRecord(g->ev1, s));
  SB_CUDA(cudaStreamSynchronize(s));
  if (h[2]) SB_FAIL(SB200_EFORMAT, "%llu queries hit the decode watchdog (inconsistent posting data)", h[2]);
  if (stats) {
    float ms = 0; cudaEventElapsedTime(&ms, g->ev0, g->ev1);
    stats->postings_scored = postings; stats->docs_scored = h[0]; stats->blocks_decoded = h[1]; stats->ms = ms; cudaEventElapsedTime(&stats->kernel_ms, g->evk0, g->evk1);
  }
  return SB200_OK;
}


// Phrase batch (bm25_phrase.cuh).  Host planning per query: absent term -> no scorer (phrase_weight.rs:53-62), the distinct
// terms sorted by doc_freq (stable) with the phrase slots pointing at them, shifts = max_offset - offset.  Candidate memory is
// sum(doc_freq of the rarest term) x (8 + 4 MAXT) B for the list + 8 B for the scored matches; slots are processed in groups
// that keep it under a budget.
static int run_phrase(sb200_segment* g, const sb200_phrase_batch* b, uint32_t* docs, float* scores, uint32_t* n_out, sb200_bm25_stats* stats) {
  NvtxRange nvtx("sb200 phrase top-k batch");
  cudaStream_t s = g->stream;
  if (!b || !b->term_ords || !b->offsets || !b->lens || !b->weights || !b->tf_cache256 || !docs || !scores || !n_out) SB_FAIL(SB200_EINVAL, "NULL argument");
  if (!g->has_positions) SB_FAIL(SB200_EINVAL, "the segment has no positions attached (PhraseQuery needs WithFreqsAndPositions, phrase_query.rs:106-118)");
  const uint32_t nq = b->n_queries, nt = b->n_terms, k = b->k;
  if (nt < 2 || nt > MAXT) SB_FAIL(SB200_ERANGE, "n_terms %u outside [2,%d]", nt, MAXT);
  if (k == 0 || k > SB200_MAX_K) SB_FAIL(SB200_ERANGE, "k %u outside [1,%d]", k, SB200_MAX_K);
  for (uint32_t q = 0; q < nq; q++) {
    if (b->lens[q] < 2 || b->lens[q] > nt) SB_FAIL(SB200_EINVAL, "query %u: phrase length %u outside [2,%u] (phrase_query.rs:49-52)", q, b->lens[q], nt);
    for (uint32_t i = 0; i < b->lens[q]; i++) {
      const uint32_t ord = b->term_ords[(size_t)q * nt + i];
      if (ord != SB200_NO_TERM && ord >= g->n_terms) SB_FAIL(SB200_EINVAL, "query %u: term ordinal %u >= %u", q, ord, g->n_terms);
    }
  }
  // plan, one slot per query that can match: [terms | nd | len | slot | shift] as u32
  std::vector<uint32_t> order, pterms, pnd, plen, pslot, pshift;
  std::vector<float> pw;
  unsigned long long postings = 0;
  for (uint32_t q = 0; q < nq; q++) {
    const uint32_t L = b->lens[q];
    const uint32_t* row = b->term_ords + (size_t)q * nt;
    bool absent = false;
    for (uint32_t i = 0; i < L; i++) { if (row[i] == SB200_NO_TERM) absent = true; else postings += g->h_df[row[i]]; }
    if (absent) continue;
    uint32_t dist[MAXT], nd = 0, slot[MAXT], maxo = 0;
    for (uint32_t i = 0; i < L; i++) {
      uint32_t x = 0; while (x < nd && dist[x] != row[i]) x++;
      if (x == nd) dist[nd++] = row[i];
      maxo = std::max(maxo, b->offsets[(size_t)q * nt + i]);
    }
    uint32_t rank[MAXT];
    for (uint32_t x = 0; x < nd; x++) rank[x] = x;
    std::stable_sort(rank, rank + nd, [&](uint32_t a, uint32_t c) { return g->h_df[dist[a]] < g->h_df[dist[c]]; });
    uint32_t where[MAXT];
    for (uint32_t x = 0; x < nd; x++) where[rank[x]] = x;
    for (uint32_t i = 0; i < L; i++) { uint32_t x = 0; while (dist[x] != row[i]) x++; slot[i] = where[x]; }
    order.push_back(q);
    for (uint32_t x = 0; x < MAXT; x++) pterms.push_back(x < nd ? dist[rank[x]] : 0u);
    pnd.push_back(nd); plen.push_back(L); pw.push_back(b->weights[q]);
    for (uint32_t i = 0; i < MAXT; i++) { pslot.push_back(i < L ? slot[i] : 0u); pshift.push_back(i < L ? maxo - b->offsets[(size_t)q * nt + i] : 0u); }
  }
  if (nq == 0) return SB200_OK;
  const uint32_t ns = (uint32_t)order.size();
  SB_TRY(ensure(g->o_docs, std::max<size_t>((size_t)nq * k, 1))); SB_TRY(ensure(g->o_scores, std::max<size_t>((size_t)nq * k, 1)));
  SB_TRY(ensure(g->o_n, std::max<uint32_t>(nq, 1))); SB_TRY(ensure(g->counters, 4)); SB_TRY(ensure(g->q_cache, 256));
  SB_TRY(ensure(g->q_orig, std::max<uint32_t>(ns, 1))); SB_TRY(ensure(g->ph_w, std::max<size_t>((size_t)ns * (MAXT + 1), 1)));
  SB_TRY(ensure(g->ph_plan, std::max<size_t>((size_t)ns * (3 * MAXT + 2), 1))); SB_TRY(ensure(g->ph_n, 1));
  SB_TRY(ensure(g->a3_off, std::max<uint32_t>(ns, 1))); SB_TRY(ensure(g->a3_cnt, std::max<uint32_t>(ns, 1)));
  uint32_t* d_terms = g->ph_plan.p; uint32_t* d_slot = d_terms + (size_t)ns * MAXT; uint32_t* d_shift = d_slot + (size_t)ns * MAXT;
  uint32_t* d_nd = d_shift + (size_t)ns * MAXT; uint32_t* d_len = d_nd + ns;
  SB_CUDA(cudaEventRecord(g->ev0, s));
  SB_CUDA(cudaMemsetAsync(g->o_n.p, 0, (size_t)std::max<uint32_t>(nq, 1) * 4, s));
  SB_CUDA(cudaMemsetAsync(g->counters.p, 0, 4 * sizeof(unsigned long long), s));
  SB_CUDA(cudaMemcpyAsync(g->q_cache.p, b->tf_cache256, 256 * 4, cudaMemcpyDefault, s));
  if (ns) {
    SB_CUDA(cudaMemcpyAsync(g->q_orig.p, order.data(), (size_t)ns * 4, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_terms, pterms.data(), pterms.size() * 4, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_slot, pslot.data(), pslot.size() * 4, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_shift, pshift.data(), pshift.size() * 4, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_nd, pnd.data(), pnd.size() * 4, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_len, plen.data(), plen.size() * 4, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(g->ph_w.p, pw.data(), pw.size() * 4, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemsetAsync(g->ph_w.p + ns, 0, (size_t)ns * MAXT * 4, s));
  }
  static size_t sel_conf = 0;
  const size_t sel_smem = (size_t)A3_SEL_CAP * 8;
  if (sel_conf < sel_smem) {
    SB_CUDA(cudaFuncSetAttribute(k_and3_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sel_smem));
    sel_conf = sel_smem;
  }
  const uint64_t max_entries = std::max<uint64_t>(((uint64_t)4 << 30) / (16 + 4 * MAXT), 1);
  std::vector<uint64_t> off(std::max<uint32_t>(ns, 1), 0);
  std::vector<AUnit> units;
  unsigned long long n_cand = 0;
  SB_CUDA(cudaEventRecord(g->evk0, s));
  uint32_t g0 = 0;
  while (g0 < ns) {
    uint64_t entries = 0; uint32_t g1 = g0;
    units.clear();
    while (g1 < ns) {
      const uint32_t dfA = g->h_df[pterms[(size_t)g1 * MAXT]];
      if (g1 > g0 && entries + dfA > max_entries) break;
      off[g1] = entries; entries += dfA;
      const uint32_t nblk = (dfA >> 7) + ((dfA & 127u) ? 1u : 0u);
      for (uint32_t b0 = 0; b0 < nblk; b0 += A3_UNIT_BLOCKS) {
        AUnit u; u.q = g1; u.blk_lo = b0; u.blk_hi = std::min(nblk, b0 + A3_UNIT_BLOCKS); u._pad = 0;
        units.push_back(u);
      }
      g1++;
    }
    const uint32_t n_units = (uint32_t)units.size();
    const size_t cap = (size_t)std::max<uint64_t>(entries, 1);
    SB_TRY(ensure(g->ph_cq, cap)); SB_TRY(ensure(g->ph_cdoc, cap)); SB_TRY(ensure(g->ph_cord, cap * MAXT));
    SB_TRY(ensure(g->a3_key, cap)); SB_TRY(ensure(g->a3_doc, cap)); SB_TRY(ensure(g->a3_units, std::max<size_t>(n_units, 1)));
    SB_CUDA(cudaMemcpyAsync(g->a3_off.p + g0, off.data() + g0, (size_t)(g1 - g0) * 8, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemsetAsync(g->a3_cnt.p + g0, 0, (size_t)(g1 - g0) * 4, s));
    SB_CUDA(cudaMemsetAsync(g->ph_n.p, 0, sizeof(unsigned long long), s));
    if (n_units) {
      SB_CUDA(cudaMemcpyAsync(g->a3_units.p, units.data(), (size_t)n_units * sizeof(AUnit), cudaMemcpyHostToDevice, s));
      PhParams PP;
      memset(&PP, 0, sizeof(PP));
      A3Params& A = PP.A;
      seg_view(g, A.S); A.a128 = g->a_post.p; A.t_aoff = g->t_aoff.p;
      A.q_terms = d_terms; A.q_nterms = d_nd; A.q_weights = g->ph_w.p + ns; A.cache = g->q_cache.p; A.n_terms_max = MAXT;
      A.units = (const AUnit*)g->a3_units.p; A.n_units = n_units; A.counters = g->counters.p;
      PP.b_pos = g->b_pos.p; PP.pa = g->pa.p; PP.pb_off = g->pb_off.p; PP.pb_bits = g->pb_bits.p;
      PP.pt_afirst = g->pt_afirst.p; PP.pt_nb = g->pt_nb.p; PP.pt_tail = g->pt_tail.p; PP.ptail = g->ptail.p; PP.pt_total = g->pt_total.p;
      PP.q_len = d_len; PP.q_slot = d_slot; PP.q_shift = d_shift; PP.q_weight = g->ph_w.p;
      PP.c_q = g->ph_cq.p; PP.c_doc = g->ph_cdoc.p; PP.c_ord = g->ph_cord.p; PP.c_n = g->ph_n.p; PP.c_cap = cap;
      PP.r_off = g->a3_off.p; PP.r_cnt = g->a3_cnt.p; PP.r_key = g->a3_key.p; PP.r_doc = g->a3_doc.p; PP.counters = g->counters.p;
      SB_LAUNCH(k_phrase_docs, div_up(n_units, A3_WARPS), A3_WARPS * 32, 0, s, PP);
      SB_CHECK_LAUNCH();
      const unsigned grid = (unsigned)std::min<uint64_t>(div_up(cap, A3_WARPS), 148u * 16u);
      SB_LAUNCH(k_phrase_match, grid, A3_WARPS * 32, 0, s, PP);
      SB_CHECK_LAUNCH();
    }
    SB_LAUNCH(k_and3_select, g1 - g0, 256, sel_smem, s, g->a3_off.p, g->a3_cnt.p, g->a3_key.p, g->a3_doc.p, g->q_orig.p, g0, k,
              g->o_docs.p, g->o_scores.p, g->o_n.p);
    SB_CHECK_LAUNCH();
    unsigned long long c = 0;
    SB_CUDA(cudaMemcpyAsync(&c, g->ph_n.p, sizeof(c), cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaStreamSynchronize(s));   // `units` / `off` are reused by the next group's async copies
    n_cand += c;
    g0 = g1;
  }
  SB_CUDA(cudaEventRecord(g->evk1, s));
  SB_TRY(copy_out_tables(g, nq, k, docs, scores, nullptr, n_out));
  unsigned long long h[4] = {0, 0, 0, 0};
  SB_CUDA(cudaMemcpyAsync(h, g->counters.p, sizeof(h), cudaMemcpyDeviceToHost, s));
  SB_CUDA(cudaEventRecord(g->ev1, s));
  SB_CUDA(cudaStreamSynchronize(s));
  if (h[2]) SB_FAIL(SB200_EFORMAT, "%llu phrase work items met inconsistent posting or position data", h[2]);
  if (stats) {
    float ms = 0; cudaEventElapsedTime(&ms, g->ev0, g->ev1);
    stats->postings_scored = postings; stats->docs_scored = n_cand; stats->blocks_decoded = h[1]; stats->ms = ms;
    cudaEventElapsedTime(&stats->kernel_ms, g->evk0, g->evk1);
  }
  return SB200_OK;
}

}  // namespace sb200
using namespace sb200;

namespace sb200 {
// TermInfoStore::get for every term ordinal (tantivy/src/termdict/fst_termdict/term_info_store.rs:55-99,134-153): the
// block's first TermInfo comes verbatim from its 47-byte TermInfoBlockMeta, the other 255 are bit-packed offsets
// relative to it, read with the reference's unaligned little-endian 8-byte window (:102-122).
__device__ __forceinline__ uint64_t tis_u64(const uint8_t* p, uint64_t avail) {
  uint64_t v = 0;
  for (uint32_t i = 0; i < 8u && i < avail; i++) v |= (uint64_t)p[i] << (8u * i);
  return v;
}
__device__ __forceinline__ uint64_t tis_bits(const uint8_t* data, uint64_t len, uint64_t addr_bits, uint32_t nb) {
  const uint64_t ab = addr_bits >> 3;
  if (ab >= len) return 0;
  const uint64_t v = tis_u64(data + ab, len - ab) >> (addr_bits & 7u);
  return v & ((1ull << nb) - 1ull);
}
__global__ void k_term_info_store(const uint8_t* __restrict__ file, uint64_t len, uint64_t meta_len, uint64_t n_terms,
                                  sb200_term_info* out, uint64_t* pos_s, uint64_t* pos_e, int* err) {
  const uint64_t ord = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (ord >= n_terms) return;
  const uint8_t* m = file + 16 + (ord >> 8) * 47;
  const uint8_t* infos = file + 16 + meta_len;
  const uint64_t infos_len = len - 16 - meta_len;
  const uint64_t off = tis_u64(m, 8);
  const uint32_t rdf = (uint32_t)tis_u64(m + 8, 4);
  const uint64_t rps = tis_u64(m + 12, 8), rpl = tis_u64(m + 20, 8);
  const uint32_t dfb = m[44], pb = m[45], qb = m[46];
  const uint32_t inner = (uint32_t)(ord & 255u);
  sb200_term_info ti; ti._pad = 0;
  if (inner == 0) {
    ti.postings_off = rps; ti.postings_len = rpl; ti.doc_freq = rdf;
    if (pos_s) { const uint64_t qs = tis_u64(m + 28, 8); pos_s[ord] = qs; pos_e[ord] = qs + tis_u64(m + 36, 8); }
  } else {
    if (off > infos_len || dfb > 56 || pb > 56 || qb > 56) { *err = 1; return; }
    const uint64_t nb = (uint64_t)dfb + pb + qb, a0 = nb * (inner - 1);
    const uint8_t* d = infos + off; const uint64_t dl = infos_len - off;
    const uint64_t ps = rps + tis_bits(d, dl, a0, pb), pe = rps + tis_bits(d, dl, a0 + nb, pb);
    if (pe < ps) { *err = 2; return; }
    ti.postings_off = ps; ti.postings_len = pe - ps;
    ti.doc_freq = (uint32_t)tis_bits(d, dl, a0 + pb + qb, dfb);
    if (pos_s) {   // positions_range: start at a0 + pb, end = the next term's start (term_info_store.rs:66-91)
      const uint64_t qs = tis_u64(m + 28, 8);
      const uint64_t s0 = qs + tis_bits(d, dl, a0 + pb, qb), s1 = qs + tis_bits(d, dl, a0 + pb + nb, qb);
      if (s1 < s0) { *err = 3; return; }
      pos_s[ord] = s0; pos_e[ord] = s1;
    }
  }
  out[ord] = ti;
}
}  // namespace sb200

extern "C" {

static int tis_decode(const uint8_t* store, uint64_t len, int device, sb200_term_info* infos, uint64_t* pos_start, uint64_t* pos_end,
                      uint64_t cap, uint64_t* n_terms) {
  using namespace sb200;
  if (!store || !n_terms) SB_FAIL(SB200_EINVAL, "NULL argument");
  if (len < 16) SB_FAIL(SB200_EFORMAT, "term info store shorter than its 16-byte header");
  SB_CUDA(cudaSetDevice(device));
  uint8_t head[16];
  SB_CUDA(cudaMemcpy(head, store, 16, cudaMemcpyDefault));
  uint64_t meta_len = 0, n = 0;
  memcpy(&meta_len, head, 8); memcpy(&n, head + 8, 8);
  if (meta_len > len - 16 || meta_len != 47ull * ((n + 255) / 256)) SB_FAIL(SB200_EFORMAT, "term info store: %llu terms need %llu bytes of block metadata, header says %llu", (unsigned long long)n, (unsigned long long)(47ull * ((n + 255) / 256)), (unsigned long long)meta_len);
  *n_terms = n;
  const uint64_t k = std::min<uint64_t>(n, cap);
  if ((!infos && !pos_start) || k == 0) return SB200_OK;
  DevBuf<uint8_t> d_store; DevBuf<sb200_term_info> d_out; DevBuf<int> d_err; DevBuf<uint64_t> d_pos;
  SB_TRY(d_store.alloc(len)); SB_TRY(d_out.alloc(n)); SB_TRY(d_err.alloc(1));
  if (pos_start) SB_TRY(d_pos.alloc(2 * n));
  SB_CUDA(cudaMemcpy(d_store.p, store, len, cudaMemcpyDefault));
  SB_CUDA(cudaMemset(d_err.p, 0, sizeof(int)));
  SB_LAUNCH(k_term_info_store, div_up(n, 256), 256, 0, (cudaStream_t)0, d_store.p, len, meta_len, n, d_out.p,
            pos_start ? d_pos.p : nullptr, pos_start ? d_pos.p + n : nullptr, d_err.p);
  SB_CHECK_LAUNCH();
  int h_err = 0;
  SB_CUDA(cudaMemcpy(&h_err, d_err.p, sizeof(int), cudaMemcpyDeviceToHost));
  if (h_err) SB_FAIL(SB200_EFORMAT, "term info store is inconsistent (code %d)", h_err);
  if (infos) SB_CUDA(cudaMemcpy(infos, d_out.p, k * sizeof(sb200_term_info), cudaMemcpyDefault));
  if (pos_start) {
    SB_CUDA(cudaMemcpy(pos_start, d_pos.p, k * 8, cudaMemcpyDefault));
    SB_CUDA(cudaMemcpy(pos_end, d_pos.p + n, k * 8, cudaMemcpyDefault));
  }
  return SB200_OK;
}

int sb200_term_info_store_decode(const uint8_t* store, uint64_t len, int device, sb200_term_info* infos, uint64_t cap,
                                 uint64_t* n_terms) {
  return tis_decode(store, len, device, infos, nullptr, nullptr, cap, n_terms);
}

int sb200_term_info_store_decode_positions(const uint8_t* store, uint64_t len, int device, uint64_t* pos_start, uint64_t* pos_end,
                                           uint64_t cap, uint64_t* n_terms) {
  if (cap && (!pos_start || !pos_end)) SB_FAIL(SB200_EINVAL, "NULL argument");
  return tis_decode(store, len, device, nullptr, cap ? pos_start : nullptr, pos_end, cap, n_terms);
}

int sb200_segment_create(const uint8_t* postings_file, uint64_t postings_len, const sb200_term_info* terms, uint32_t n_terms,
                         const uint8_t* fieldnorm_ids, uint32_t max_doc, int record_option, int device, sb200_segment** out) {
  if (!out) SB_FAIL(SB200_EINVAL, "out is NULL");
  *out = nullptr;
  if ((postings_len && !postings_file) || (n_terms && !terms) || (max_doc && !fieldnorm_ids)) SB_FAIL(SB200_EINVAL, "NULL argument");
  if (record_option < 0 || record_option > 2) SB_FAIL(SB200_EINVAL, "record_option %d", record_option);
  if (max_doc >= TERMINATED) SB_FAIL(SB200_ERANGE, "max_doc must be < 2^31-1 (TERMINATED, tantivy/src/docset.rs:9)");
  int ndev = 0;
  SB_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) SB_FAIL(SB200_EINVAL, "device %d not in [0,%d)", device, ndev);
  SB_CUDA(cudaSetDevice(device));
  sb200_segment* g = new (std::nothrow) sb200_segment();
  if (!g) SB_FAIL(SB200_ENOMEM, "host allocation failed");
  g->device = device; g->record = record_option; g->stride = record_option == 0 ? 5 : (record_option == 1 ? 8 : 12);
  g->max_doc = max_doc; g->n_terms = n_terms; g->postings_len = postings_len;
  auto body = [&]() -> int {
    SB_CUDA(cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking));
    SB_CUDA(cudaEventCreate(&g->ev0)); SB_CUDA(cudaEventCreate(&g->ev1));
    SB_CUDA(cudaEventCreate(&g->evk0)); SB_CUDA(cudaEventCreate(&g->evk1));
    cudaStream_t s = g->stream;
    SB_CUDA(cudaEventRecord(g->ev0, s));
    SB_TRY(g->postings.alloc(postings_len + 64));
    SB_CUDA(cudaMemsetAsync(g->postings.p + postings_len, 0, 64, s));
    SB_TRY(copy_in(g->postings.p, postings_file, postings_len, s));
    SB_TRY(g->fieldnorm.alloc((size_t)max_doc + 16));
    SB_TRY(copy_in(g->fieldnorm.p, fieldnorm_ids, max_doc, s));
    // block slots: n_full + 1 per term (the extra one records where the vint tail starts)
    std::vector<sb200_term_info> h_terms;
    const sb200_term_info* ht = terms;
    if (n_terms && is_device_ptr(terms)) { h_terms.resize(n_terms); SB_CUDA(cudaMemcpy(h_terms.data(), terms, (size_t)n_terms * sizeof(sb200_term_info), cudaMemcpyDeviceToHost)); ht = h_terms.data(); }
    std::vector<uint32_t> first(n_terms + 1);
    g->h_df.resize(n_terms);
    uint64_t slots = 0, postings = 0;
    for (uint32_t t = 0; t < n_terms; t++) {
      first[t] = (uint32_t)slots; slots += (ht[t].doc_freq >> 7) + 1; g->h_df[t] = ht[t].doc_freq; postings += ht[t].doc_freq;
      if (slots >= 0xFFFFFFF0ull) SB_FAIL(SB200_ERANGE, "more than 2^32 posting blocks");
      if (ht[t].postings_len >= 0xFFFFFFFFull) SB_FAIL(SB200_ERANGE, "term %u: posting list larger than 4 GiB", t);
    }
    first[n_terms] = (uint32_t)slots;
    g->n_blocks = slots - n_terms; g->n_postings = postings;
    SB_TRY(g->t_first.alloc(n_terms + 1)); SB_TRY(g->t_data_off.alloc(n_terms + 1)); SB_TRY(g->t_end_off.alloc(n_terms + 1)); SB_TRY(g->t_df.alloc(n_terms + 1));
    SB_TRY(g->b_last.alloc(slots + 1)); SB_TRY(g->b_off.alloc(slots + 1)); SB_TRY(g->b_bits.alloc(slots + 1)); SB_TRY(g->b_bw.alloc(slots + 1));
    SB_CUDA(cudaMemcpyAsync(g->t_first.p, first.data(), (size_t)(n_terms + 1) * 4, cudaMemcpyHostToDevice, s));
    DevBuf<sb200_term_info> d_terms; DevBuf<int> d_err;
    SB_TRY(d_terms.alloc(n_terms + 1)); SB_TRY(d_err.alloc(1));
    SB_CUDA(cudaMemcpyAsync(d_terms.p, ht, (size_t)n_terms * sizeof(sb200_term_info), cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemsetAsync(d_err.p, 0, sizeof(int), s));
    if (n_terms) {
      SB_LAUNCH(k_build_directory, div_up((uint64_t)n_terms * 32, 256), 256, 0, s, g->postings.p, d_terms.p, n_terms, g->stride,
                g->t_first.p, g->t_data_off.p, g->t_end_off.p, g->t_df.p, g->b_last.p, g->b_off.p, g->b_bits.p, g->b_bw.p, postings_len, d_err.p);
      SB_CHECK_LAUNCH();
    }
    int h_err = 0;
    SB_CUDA(cudaMemcpyAsync(&h_err, d_err.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaStreamSynchronize(s));
    if (h_err) SB_FAIL(SB200_EFORMAT, "malformed postings (code %d): term range outside the file, skip length != blocks x %d, or bit width > 32", h_err, g->stride);
    // aligned copy of the block regions: per-term size (uint4 units) -> exclusive scan -> realigning copy
    SB_TRY(g->t_aoff.alloc(n_terms + 1));
    uint64_t total_units = 0;
    if (n_terms) {
      DevBuf<uint64_t> units; SB_TRY(units.alloc(n_terms + 1));
      SB_CUDA(cudaMemsetAsync(units.p + n_terms, 0, 8, s));
      SB_LAUNCH(k_block_units, div_up(n_terms, 256), 256, 0, s, g->t_first.p, g->t_df.p, g->b_off.p, n_terms, units.p);
      SB_CHECK_LAUNCH();
      size_t need = 0;
      SB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, need, units.p, g->t_aoff.p, (int64_t)(n_terms + 1), s));
      DevBuf<uint8_t> tmp; SB_TRY(tmp.alloc(need + 256));
      SB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, need, units.p, g->t_aoff.p, (int64_t)(n_terms + 1), s));
      g_launches.fetch_add(2, std::memory_order_relaxed);
      SB_CUDA(cudaMemcpyAsync(&total_units, g->t_aoff.p + n_terms, 8, cudaMemcpyDeviceToHost, s));
      SB_CUDA(cudaStreamSynchronize(s));
    }
    SB_TRY(g->a_post.alloc(total_units + 4));
    if (n_terms && total_units) {
      SB_LAUNCH(k_align_blocks, div_up((uint64_t)n_terms * 32, 256), 256, 0, s, (const uint32_t*)g->postings.p, g->t_data_off.p,
                g->t_first.p, g->t_df.p, g->b_off.p, g->t_aoff.p, n_terms, (uint32_t*)g->a_post.p);
      SB_CHECK_LAUNCH();
    }
    SB_CUDA(cudaEventRecord(g->ev1, s));
    SB_CUDA(cudaStreamSynchronize(s));
    float ms = 0; cudaEventElapsedTime(&ms, g->ev0, g->ev1); g->stage_ms = ms;
    return SB200_OK;
  };
  const int rc = body();
  if (rc != SB200_OK) { sb200_segment_destroy(g); return rc; }
  *out = g;
  return SB200_OK;
}

void sb200_segment_destroy(sb200_segment* g) {
  if (!g) return;
  cudaSetDevice(g->device);
  if (g->stream) cudaStreamSynchronize(g->stream);
  if (g->ev0) cudaEventDestroy(g->ev0);
  if (g->ev1) cudaEventDestroy(g->ev1);
  if (g->evk0) cudaEventDestroy(g->evk0);
  if (g->evk1) cudaEventDestroy(g->evk1);
  if (g->h_pack) cudaFreeHost(g->h_pack);
  cudaStream_t s = g->stream;
  delete g;
  if (s) cudaStreamDestroy(s);
}

int sb200_segment_get_info(const sb200_segment* g, sb200_segment_info* info) {
  if (!g || !info) SB_FAIL(SB200_EINVAL, "NULL argument");
  info->n_terms = g->n_terms; info->n_blocks = g->n_blocks; info->n_postings = g->n_postings; info->max_doc = g->max_doc; info->_pad = 0;
  info->hbm_bytes = g->postings.bytes() + g->fieldnorm.bytes() + g->t_first.bytes() + g->t_data_off.bytes() + g->t_end_off.bytes() +
                    g->t_df.bytes() + g->b_last.bytes() + g->b_off.bytes() + g->b_bits.bytes() + g->b_bw.bytes() +
                    g->pos_file.bytes() + g->pb_bits.bytes() + g->b_pos.bytes() + g->pt_total.bytes() + g->pt_afirst.bytes() +
                    g->pt_tail.bytes() + g->pb_off.bytes() + g->pt_nb.bytes() + g->ptail.bytes() + g->pa.bytes();
  info->stage_ms = g->stage_ms;
  return SB200_OK;
}

int sb200_signals_create(const double* const* columns, uint32_t n_cols, uint32_t max_doc, int device, sb200_signals** out) {
  if (!out) SB_FAIL(SB200_EINVAL, "out is NULL");
  *out = nullptr;
  if (n_cols && !columns) SB_FAIL(SB200_EINVAL, "columns is NULL");
  if (n_cols > 64) SB_FAIL(SB200_ERANGE, "at most 64 signal columns");
  SB_CUDA(cudaSetDevice(device));
  sb200_signals* sg = new (std::nothrow) sb200_signals();
  if (!sg) SB_FAIL(SB200_ENOMEM, "host allocation failed");
  sg->device = device; sg->n_cols = n_cols; sg->max_doc = max_doc;
  auto body = [&]() -> int {
    if (!n_cols || !max_doc) return SB200_OK;
    SB_TRY(sg->rows.alloc((size_t)max_doc * n_cols));
    std::vector<DevBuf<double>> tmp(n_cols);
    std::vector<const double*> ptrs(n_cols);
    for (uint32_t c = 0; c < n_cols; c++) {
      if (!columns[c]) SB_FAIL(SB200_EINVAL, "column %u is NULL", c);
      if (is_device_ptr(columns[c])) ptrs[c] = columns[c];
      else { SB_TRY(tmp[c].alloc(max_doc)); SB_CUDA(cudaMemcpy(tmp[c].p, columns[c], (size_t)max_doc * 8, cudaMemcpyHostToDevice)); ptrs[c] = tmp[c].p; }
    }
    DevBuf<const double*> d_ptrs; SB_TRY(d_ptrs.alloc(n_cols));
    SB_CUDA(cudaMemcpy(d_ptrs.p, ptrs.data(), n_cols * sizeof(double*), cudaMemcpyHostToDevice));
    SB_LAUNCH(k_interleave_signals, div_up((uint64_t)max_doc * n_cols, 256), 256, 0, 0, d_ptrs.p, n_cols, max_doc, sg->rows.p);
    SB_CHECK_LAUNCH();
    SB_CUDA(cudaDeviceSynchronize());
    return SB200_OK;
  };
  const int rc = body();
  if (rc != SB200_OK) { delete sg; return rc; }
  *out = sg;
  return SB200_OK;
}
int sb200_signals_create_raw(const sb200_numeric_column* cols, uint32_t n_cols, uint32_t max_doc, int device, sb200_signals** out) {
  if (!out) SB_FAIL(SB200_EINVAL, "out is NULL");
  *out = nullptr;
  if (n_cols && !cols) SB_FAIL(SB200_EINVAL, "cols is NULL");
  if (n_cols > 64) SB_FAIL(SB200_ERANGE, "at most 64 signal columns");
  SB_CUDA(cudaSetDevice(device));
  sb200_signals* sg = new (std::nothrow) sb200_signals();
  if (!sg) SB_FAIL(SB200_ENOMEM, "host allocation failed");
  sg->device = device; sg->n_cols = n_cols; sg->max_doc = max_doc;
  auto body = [&]() -> int {
    if (!n_cols || !max_doc) return SB200_OK;
    SB_TRY(sg->rows.alloc((size_t)max_doc * n_cols));
    for (uint32_t c = 0; c < n_cols; c++) {
      const sb200_numeric_column& col = cols[c];
      if (!col.raw) SB_FAIL(SB200_EINVAL, "column %u: raw is NULL", c);
      if (col.dtype > SB200_NUM_BOOL8) SB_FAIL(SB200_EINVAL, "column %u: unknown dtype %u", c, col.dtype);
      if (col.kind > SB200_NUM_REGION) SB_FAIL(SB200_EINVAL, "column %u: unknown transform %u", c, col.kind);
      const size_t esz = col.dtype == SB200_NUM_BOOL8 ? 1 : 8;
      DevBuf<uint8_t> d_raw; DevBuf<double> d_lut;
      if (col.kind == SB200_NUM_RANK) {
        // score_rank = (10 - (1 + rank).log(8)).max(0) (non_text.rs:50-59), f64::log(base) = ln(x) / ln(base).  `ln` is the host
        // C library's (as for a Rust binary on the same machine); no device `log` is bit-identical to it, so this one transform
        // is evaluated on the host at open time and only the finished column crosses PCIe.
        if (col.dtype != SB200_NUM_U64) SB_FAIL(SB200_EINVAL, "column %u: score_rank reads a u64 column", c);
        std::vector<uint64_t> h_raw;
        const uint64_t* r = (const uint64_t*)col.raw;
        if (is_device_ptr(col.raw)) { h_raw.resize(max_doc); SB_CUDA(cudaMemcpy(h_raw.data(), col.raw, (size_t)max_doc * 8, cudaMemcpyDeviceToHost)); r = h_raw.data(); }
        std::vector<double> sc(max_doc);
        const double ln8 = log(8.0);
        for (uint32_t d = 0; d < max_doc; d++) { const double v = 10.0 - log(1.0 + (double)r[d]) / ln8; sc[d] = v > 0.0 ? v : 0.0; }
        SB_TRY(d_raw.alloc((size_t)max_doc * 8));
        SB_CUDA(cudaMemcpy(d_raw.p, sc.data(), (size_t)max_doc * 8, cudaMemcpyHostToDevice));
        SB_LAUNCH(k_numeric_score, div_up(max_doc, 256), 256, 0, 0, (uint32_t)SB200_NUM_IDENTITY, (uint32_t)SB200_NUM_F64, (const void*)d_raw.p, max_doc, 0.0, 0.0,
                  (const double*)nullptr, 0u, sg->rows.p, n_cols, c);
        SB_CHECK_LAUNCH();
        SB_CUDA(cudaDeviceSynchronize());
        continue;
      }
      const void* raw = col.raw;
      if (!is_device_ptr(col.raw)) {
        SB_TRY(d_raw.alloc((size_t)max_doc * esz));
        SB_CUDA(cudaMemcpy(d_raw.p, col.raw, (size_t)max_doc * esz, cudaMemcpyHostToDevice));
        raw = d_raw.p;
      }
      const double* lut = nullptr;
      if (col.kind == SB200_NUM_REGION && col.lut && col.lut_len) {
        SB_TRY(d_lut.alloc(col.lut_len));
        SB_CUDA(cudaMemcpy(d_lut.p, col.lut, (size_t)col.lut_len * 8, cudaMemcpyDefault));
        lut = d_lut.p;
      }
      SB_LAUNCH(k_numeric_score, div_up(max_doc, 256), 256, 0, 0, col.kind, col.dtype, raw, max_doc, col.p0, col.p1, lut, lut ? col.lut_len : 0u,
                sg->rows.p, n_cols, c);
      SB_CHECK_LAUNCH();
      SB_CUDA(cudaDeviceSynchronize());   // the staging copies of this column are released at the end of the iteration
    }
    return SB200_OK;
  };
  const int rc = body();
  if (rc != SB200_OK) { delete sg; return rc; }
  *out = sg;
  return SB200_OK;
}
int sb200_signals_read(const sb200_signals* s, uint32_t first_doc, uint32_t n_docs, double* rows_out) {
  if (!s || (!rows_out && n_docs)) SB_FAIL(SB200_EINVAL, "NULL argument");
  if ((uint64_t)first_doc + n_docs > s->max_doc) SB_FAIL(SB200_ERANGE, "docs [%u, +%u) outside the table of %u", first_doc, n_docs, s->max_doc);
  SB_CUDA(cudaSetDevice(s->device));
  if (n_docs && s->n_cols)
    SB_CUDA(cudaMemcpy(rows_out, s->rows.p + (size_t)first_doc * s->n_cols, (size_t)n_docs * s->n_cols * 8, cudaMemcpyDeviceToHost));
  return SB200_OK;
}
void sb200_signals_destroy(sb200_signals* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  delete s;
}

int sb200_segment_attach_positions(sb200_segment* g, const uint8_t* positions_file, uint64_t len, const uint64_t* pos_start,
                                   const uint64_t* pos_end) {
  if (!g) SB_FAIL(SB200_EINVAL, "NULL segment handle");
  if (g->record != SB200_RECORD_FREQS_POSITIONS) SB_FAIL(SB200_EINVAL, "positions need a WithFreqsAndPositions segment (record option 2), this one has %d", g->record);
  if ((len && !positions_file) || (g->n_terms && (!pos_start || !pos_end))) SB_FAIL(SB200_EINVAL, "NULL argument");
  SB_CUDA(cudaSetDevice(g->device));
  const uint32_t nt = g->n_terms;
  std::vector<uint64_t> hs(nt), he(nt);
  if (nt) {
    SB_CUDA(cudaMemcpy(hs.data(), pos_start, (size_t)nt * 8, cudaMemcpyDefault));
    SB_CUDA(cudaMemcpy(he.data(), pos_end, (size_t)nt * 8, cudaMemcpyDefault));
  }
  for (uint32_t t = 0; t < nt; t++)
    if (hs[t] > he[t] || he[t] > len) SB_FAIL(SB200_EFORMAT, "term %u: positions range [%llu, %llu) outside the %llu-byte file", t,
                                              (unsigned long long)hs[t], (unsigned long long)he[t], (unsigned long long)len);
  g->has_positions = false;
  cudaStream_t s = g->stream;
  auto body = [&]() -> int {
    SB_TRY(g->pos_file.alloc(len + 64));
    SB_CUDA(cudaMemsetAsync(g->pos_file.p + len, 0, 64, s));
    if (len) SB_TRY(copy_in(g->pos_file.p, positions_file, len, s));
    const size_t slots = g->b_last.n;
    SB_TRY(g->b_pos.alloc(slots)); SB_TRY(g->pt_total.alloc(nt + 1)); SB_TRY(g->pt_nb.alloc(nt + 1));
    DevBuf<uint64_t> d_se, d_hdr, d_packed, d_au; DevBuf<int> d_err;
    SB_TRY(d_se.alloc(2 * (size_t)nt + 2)); SB_TRY(d_hdr.alloc(nt + 1)); SB_TRY(d_packed.alloc(nt + 1)); SB_TRY(d_err.alloc(1));
    SB_CUDA(cudaMemcpyAsync(d_se.p, hs.data(), (size_t)nt * 8, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_se.p + nt, he.data(), (size_t)nt * 8, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemsetAsync(d_err.p, 0, sizeof(int), s));
    if (nt) {
      SB_LAUNCH(k_pos_scan, div_up((uint64_t)nt * 32, 256), 256, 0, s, g->postings.p, g->t_first.p, g->t_df.p, g->t_data_off.p, g->t_end_off.p,
                g->b_off.p, nt, g->pos_file.p, d_se.p, d_se.p + nt, g->b_pos.p, g->pt_total.p, g->pt_nb.p, d_hdr.p, d_packed.p, d_err.p);
      SB_CHECK_LAUNCH();
    }
    int h_err = 0;
    SB_CUDA(cudaMemcpyAsync(&h_err, d_err.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    std::vector<uint64_t> total(nt), packed(nt); std::vector<uint32_t> nb(nt);
    if (nt) {
      SB_CUDA(cudaMemcpyAsync(total.data(), g->pt_total.p, (size_t)nt * 8, cudaMemcpyDeviceToHost, s));
      SB_CUDA(cudaMemcpyAsync(packed.data(), d_packed.p, (size_t)nt * 8, cudaMemcpyDeviceToHost, s));
      SB_CUDA(cudaMemcpyAsync(nb.data(), g->pt_nb.p, (size_t)nt * 4, cudaMemcpyDeviceToHost, s));
    }
    SB_CUDA(cudaStreamSynchronize(s));
    if (h_err) SB_FAIL(SB200_EFORMAT, "malformed positions (code %d): bad block count or vint, block count != term frequency sum / 128, "
                                      "bit width > 32, blocks past the term's range, or a tail that is not term frequency sum %% 128 vints", h_err);
    std::vector<uint64_t> afirst(nt + 1), aunits(nt + 1), tail(nt + 1);
    uint64_t a = 0, u = 0, tl = 0;
    for (uint32_t t = 0; t < nt; t++) { afirst[t] = a; aunits[t] = u; tail[t] = tl; a += nb[t]; u += packed[t] >> 4; tl += total[t] & 127u; }
    SB_TRY(g->pt_afirst.alloc(nt + 1)); SB_TRY(g->pt_tail.alloc(nt + 1)); SB_TRY(d_au.alloc(nt + 1));
    SB_TRY(g->pb_off.alloc(a + 1)); SB_TRY(g->pb_bits.alloc(a + 1)); SB_TRY(g->pa.alloc(u + 1)); SB_TRY(g->ptail.alloc(tl + 1));
    if (nt) {
      SB_CUDA(cudaMemcpyAsync(g->pt_afirst.p, afirst.data(), (size_t)nt * 8, cudaMemcpyHostToDevice, s));
      SB_CUDA(cudaMemcpyAsync(g->pt_tail.p, tail.data(), (size_t)nt * 8, cudaMemcpyHostToDevice, s));
      SB_CUDA(cudaMemcpyAsync(d_au.p, aunits.data(), (size_t)nt * 8, cudaMemcpyHostToDevice, s));
      SB_LAUNCH(k_pos_build, div_up((uint64_t)nt * 32, 256), 256, 0, s, g->pos_file.p, nt, d_hdr.p, g->pt_nb.p, d_packed.p, g->pt_total.p,
                g->pt_afirst.p, d_au.p, g->pt_tail.p, g->pb_off.p, g->pb_bits.p, (uint32_t*)g->pa.p, g->ptail.p);
      SB_CHECK_LAUNCH();
    }
    SB_CUDA(cudaStreamSynchronize(s));
    return SB200_OK;
  };
  const int rc = body();
  if (rc != SB200_OK) {
    g->pos_file.release(); g->pb_bits.release(); g->b_pos.release(); g->pt_total.release(); g->pt_afirst.release(); g->pt_tail.release();
    g->pb_off.release(); g->pt_nb.release(); g->ptail.release(); g->pa.release();
    return rc;
  }
  g->has_positions = true;
  return SB200_OK;
}

int sb200_phrase_topk_batch(sb200_segment* seg, const sb200_phrase_batch* batch, uint32_t* docs, float* scores, uint32_t* n_out,
                            sb200_bm25_stats* stats) {
  if (!seg) SB_FAIL(SB200_EINVAL, "NULL segment handle");
  SB_CUDA(cudaSetDevice(seg->device));
  return run_phrase(seg, batch, docs, scores, n_out, stats);
}

int sb200_bm25_topk_batch(sb200_segment* seg, const sb200_bm25_batch* batch, uint32_t* docs, float* scores, uint32_t* n_out,
                          sb200_bm25_stats* stats) {
  if (!seg) SB_FAIL(SB200_EINVAL, "NULL segment handle");
  SB_CUDA(cudaSetDevice(seg->device));
  if (!scores) SB_FAIL(SB200_EINVAL, "scores is NULL");
  if (!batch) SB_FAIL(SB200_EINVAL, "batch is NULL");
  return run_batch(seg, batch, batch->mode, nullptr, docs, scores, nullptr, n_out, stats);
}

int sb200_bm25_topk(sb200_segment* seg, const uint32_t* term_ords, const float* weights, uint32_t n_terms, const float* tf_cache256,
                    int mode, uint32_t k, uint32_t* docs, float* scores, uint32_t* n_out) {
  sb200_bm25_batch b;
  b.n_queries = 1; b.n_terms = n_terms; b.term_ords = term_ords; b.weights = weights; b.tf_cache256 = tf_cache256; b.mode = mode; b.k = k;
  return sb200_bm25_topk_batch(seg, &b, docs, scores, n_out, nullptr);
}

int sb200_multi_signal_topk_batch(const sb200_multi_signal_batch* batch, uint32_t* docs, double* totals, uint32_t* n_out,
                                  sb200_bm25_stats* stats) {
  return run_multi(batch, docs, totals, n_out, stats);
}
int sb200_signal_topk_batch(sb200_segment* seg, const sb200_signal_batch* batch, uint32_t* docs, double* totals, uint32_t* n_out,
                            sb200_bm25_stats* stats) {
  if (!seg) SB_FAIL(SB200_EINVAL, "NULL segment handle");
  SB_CUDA(cudaSetDevice(seg->device));
  if (!batch || !totals) SB_FAIL(SB200_EINVAL, "NULL argument");
  return run_batch(seg, &batch->q, SB200_MODE_OR, batch, docs, nullptr, totals, n_out, stats);
}

}  // extern "C"
