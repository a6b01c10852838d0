// bm25_phrase.cuh -- phrase queries with slop 0 (tantivy PhraseQuery / PhraseScorer, query/phrase_query/*.rs) over a
// segment whose positions file is attached (sb200_segment_attach_positions).
//
// Positions in HBM (built at attach time, k_pos_scan + k_pos_build):
//   b_pos      per posting block slot (first + j, incl. the tail slot first + nfull): position index of its first posting,
//              the u64 prefix sum of the 12-byte skip entries' tf_sum (skip.rs:217-232, what SkipReader::position_offset
//              accumulates, skip.rs:244-266)
//   pb_off/bits  per 128-position block of every term: its place in `pa` (uint4 units) and its bit width
//   pa         16-byte aligned copy of every term's bitpacked region (the VInt + width prefix leaves it unaligned)
//   ptail      every term's vint tail (< 128 deltas), decoded once, so a position delta is one indexed read
//   pt_total   per term: number of positions (= Σtf); every device read of the term stays below it
// Query, two kernels and the AND path's selection:
//   k_phrase_docs   the intersection of the phrase's distinct terms, exactly k_and3's unit scheme (units = query x 4 blocks
//                   of the rarest term, probes through the block directory), but instead of a score every surviving doc
//                   records, per distinct term, the ordinal of its posting (block * 128 + index) in a candidate list
//   k_phrase_match  one warp per candidate: a posting's position index is b_pos of its block plus the warp-scanned tfs
//                   before it; the count of compute_phrase_match + intersection_count (phrase_scorer.rs:435-505) with slop
//                   0 is |∩_i (positions_i + max_offset - offset_i)|.  Every per-doc list is strictly increasing, so the
//                   count does not depend on the order Intersection::new puts the terms in: the term with the smallest tf
//                   drives, 32 of its positions at a time (one per lane), and every other slot is walked as a merge in
//                   32-position chunks (a chunk is decoded by one read per lane + a warp scan; membership is a 5-step
//                   shuffle search), so long documents are chunked, never truncated.  count > 0 scores
//                   weight * (count / (count + cache[fieldnorm id])) (Bm25Weight::score, bm25.rs:182-196; PhraseScorer::score,
//                   phrase_scorer.rs:540-549) with a3_term_score's rounding
//   k_and3_select   exact top-k per query (score desc, doc asc)
#pragma once

namespace sb200 {

struct PhParams {
  A3Params A;                 // q_terms = distinct terms per query slot (doc_freq ascending), q_nterms = their number
  const uint64_t* b_pos;
  const uint4* pa; const uint64_t* pb_off; const uint8_t* pb_bits;
  const uint64_t* pt_afirst; const uint32_t* pt_nb; const uint64_t* pt_tail; const uint32_t* ptail; const uint64_t* pt_total;
  const uint32_t* q_len;      // [slot] phrase length
  const uint32_t* q_slot;     // [slot][MAXT] phrase term -> index of its distinct term
  const uint32_t* q_shift;    // [slot][MAXT] max_offset - offset
  const float* q_weight;      // [slot]
  uint32_t* c_q; uint32_t* c_doc; uint32_t* c_ord; unsigned long long* c_n; uint64_t c_cap;   // candidates, c_ord [e][MAXT]
  const uint64_t* r_off; uint32_t* r_cnt; uint32_t* r_key; uint32_t* r_doc;                  // per slot: scored matches
  unsigned long long* counters;
};

// ---- attach: validation + directories -----------------------------------------------------------------------------------
// one warp per term.  Postings side: b_pos from the skip entries, the tail's tfs from its vints -> the term's position count P.
// Positions side (positions/mod.rs:22-30, reader.rs:43-56): VInt(#blocks) == P / 128, widths <= 32, the blocks inside the range,
// and exactly P % 128 vints filling the rest of it (uncompress_vint_unsorted_until_end reads to the end of the range).
__global__ void k_pos_scan(const uint8_t* __restrict__ postings, const uint32_t* __restrict__ t_first, const uint32_t* __restrict__ t_df,
                           const uint64_t* __restrict__ t_data_off, const uint64_t* __restrict__ t_end_off, const uint32_t* __restrict__ b_off,
                           uint32_t n_terms, const uint8_t* __restrict__ pos, const uint64_t* __restrict__ pos_s,
                           const uint64_t* __restrict__ pos_e, uint64_t* b_pos, uint64_t* pt_total, uint32_t* pt_nb, uint64_t* pt_hdr,
                           uint64_t* pt_packed, int* err) {
  const uint32_t t = (blockIdx.x * (uint32_t)blockDim.x + threadIdx.x) >> 5;
  if (t >= n_terms) return;
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t df = t_df[t], nfull = df >> 7, first = t_first[t];
  const uint64_t data_off = t_data_off[t], skip0 = data_off - (uint64_t)nfull * 12u;
  uint64_t run = 0;
  for (uint32_t base = 0; base < nfull; base += 32) {
    const uint32_t j = base + lane;
    uint64_t v = 0;
    if (j < nfull) { const uint8_t* e = postings + skip0 + (uint64_t)j * 12u + 6u; v = (uint32_t)e[0] | ((uint32_t)e[1] << 8) | ((uint32_t)e[2] << 16) | ((uint32_t)e[3] << 24); }
    uint64_t incl = v;
    for (int o = 1; o < 32; o <<= 1) { const uint64_t n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
    if (j < nfull) b_pos[first + j] = run + incl - v;
    run += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) b_pos[first + nfull] = run;
  // the widths: lane-parallel; the header and both vint tails: lane 0
  uint64_t hdr = 0, P = 0; uint32_t nb = 0; int code = 0;
  if (lane == 0) {
    const uint32_t n = df & 127u;
    uint64_t p = data_off + b_off[first + nfull];
    const uint64_t end = t_end_off[t];
    uint64_t tail_tf = 0;
    for (uint32_t i = 0; i < 2 * n && !code; i++) {
      uint32_t v = 0, sh = 0; bool closed = false;
      for (int b = 0; b < 5 && p < end; b++) { const uint8_t c = postings[p++]; v |= (uint32_t)(c & 127u) << sh; sh += 7; if (c & 128u) { closed = true; break; } }
      if (!closed) code = 11;
      if (i >= n) tail_tf += v;
    }
    P = run + tail_tf;
    const uint64_t s = pos_s[t], e = pos_e[t];
    uint64_t q = s, cnt = 0; uint32_t sh = 0; bool closed = false;
    for (int b = 0; b < 10 && q < e; b++) { const uint8_t c = pos[q++]; cnt |= (uint64_t)(c & 127u) << sh; sh += 7; if (c & 128u) { closed = true; break; } }
    if (!code && !closed) code = 12;
    if (!code && cnt != (P >> 7)) code = 13;
    if (!code && cnt > e - q) code = 14;
    nb = (uint32_t)cnt; hdr = q;
    if (code) nb = 0;
  }
  nb = __shfl_sync(0xffffffffu, nb, 0); hdr = __shfl_sync(0xffffffffu, hdr, 0);
  code = __shfl_sync(0xffffffffu, code, 0);
  uint64_t packed = 0; bool wide = false;
  for (uint32_t j = lane; j < nb; j += 32) { const uint32_t w = pos[hdr + j]; wide |= w > 32; packed += (uint64_t)w * 16u; }
  for (int o = 16; o; o >>= 1) packed += __shfl_xor_sync(0xffffffffu, packed, o);
  if (__any_sync(0xffffffffu, wide) && !code) code = 15;
  if (lane == 0) {
    const uint64_t e = pos_e[t];
    const uint64_t pstart = hdr + nb;
    if (!code && packed > e - pstart) code = 16;
    if (!code) {   // the vint tail: exactly P % 128 values, the last one closed at the end of the range
      uint64_t p = pstart + packed, vals = 0;
      if (e - p > 127u * 5u) code = 17;
      while (!code && p < e) {
        bool closed = false;
        for (int b = 0; b < 5 && p < e; b++) { if (pos[p++] & 128u) { closed = true; break; } }
        if (!closed) code = 18;
        vals++;
      }
      if (!code && vals != (P & 127u)) code = 19;
    }
    pt_total[t] = code ? 0 : P; pt_nb[t] = code ? 0 : nb; pt_hdr[t] = pstart; pt_packed[t] = code ? 0 : packed;
    if (code) *err = code;   // any failing term fails the attach
  }
}

// one warp per term: the block directory, the aligned copy of the bitpacked region, the decoded vint tail
__global__ void k_pos_build(const uint8_t* __restrict__ pos, uint32_t n_terms, const uint64_t* __restrict__ pt_hdr,
                            const uint32_t* __restrict__ pt_nb, const uint64_t* __restrict__ pt_packed, const uint64_t* __restrict__ pt_total,
                            const uint64_t* __restrict__ pt_afirst, const uint64_t* __restrict__ pt_aunits, const uint64_t* __restrict__ pt_tail,
                            uint64_t* pb_off, uint8_t* pb_bits, uint32_t* pa32, uint32_t* ptail) {
  const uint32_t t = (blockIdx.x * (uint32_t)blockDim.x + threadIdx.x) >> 5;
  if (t >= n_terms) return;
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t nb = pt_nb[t];
  const uint64_t hdr = pt_hdr[t], af = pt_afirst[t], au = pt_aunits[t];
  uint64_t run = au;
  for (uint32_t base = 0; base < nb; base += 32) {
    const uint32_t j = base + lane;
    const uint32_t w = j < nb ? pos[hdr - nb + j] : 0u;
    uint32_t incl = w;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
    if (j < nb) { pb_bits[af + j] = (uint8_t)w; pb_off[af + j] = run + incl - w; }   // a block of width w is w uint4s
    run += __shfl_sync(0xffffffffu, incl, 31);
  }
  const uint64_t nbytes = pt_packed[t];
  const uint32_t* p32 = (const uint32_t*)pos;
  const uint64_t w0 = hdr >> 2; const uint32_t sh = (uint32_t)(hdr & 3u) * 8u;
  uint32_t* d = pa32 + au * 4;
  for (uint64_t w = lane; w < (nbytes >> 2); w += 32) d[w] = __funnelshift_r(__ldg(p32 + w0 + w), __ldg(p32 + w0 + w + 1), sh);
  if (lane == 0) {
    const uint32_t n = (uint32_t)(pt_total[t] & 127u);
    uint64_t p = hdr + nbytes;
    for (uint32_t i = 0; i < n; i++) {
      uint32_t v = 0, s = 0;
      for (int b = 0; b < 5; b++) { const uint8_t c = pos[p++]; v |= (uint32_t)(c & 127u) << s; s += 7; if (c & 128u) break; }
      ptail[pt_tail[t] + i] = v;
    }
  }
}

// ---- query ----------------------------------------------------------------------------------------------------------------
// position delta number p (0 <= p < pt_total[t]) of term t
__device__ __forceinline__ uint32_t ph_delta(const PhParams& P, uint32_t t, uint64_t p) {
  const uint64_t nb = P.pt_nb[t];
  if (p < nb * 128u) {
    const uint64_t a = P.pt_afirst[t] + (p >> 7);
    const uint32_t w = P.pb_bits[a], k = (uint32_t)(p & 127u);
    if (w == 0) return 0;
    const uint32_t* words = (const uint32_t*)(P.pa + P.pb_off[a]);
    const uint32_t l4 = k & 3u, bit = (k >> 2) * w, wi = bit >> 5, sh = bit & 31u;
    const uint32_t lo = __ldg(words + wi * 4 + l4);
    const uint32_t hi = (sh + w > 32) ? __ldg(words + (wi + 1) * 4 + l4) : 0u;
    const uint32_t v = __funnelshift_r(lo, hi, sh);
    return w == 32 ? v : (v & ((1u << w) - 1u));
  }
  return __ldg(P.ptail + P.pt_tail[t] + (p - nb * 128u));
}

// The intersection of k_and3 over a query slot's distinct terms; a surviving doc goes to the candidate list with the posting
// ordinal of every distinct term (kept in shared memory while the later terms are probed).
__global__ void __launch_bounds__(A3_WARPS * 32) k_phrase_docs(const PhParams PP) {
  __shared__ __align__(16) uint32_t s_docs[A3_WARPS][128];
  __shared__ __align__(16) uint32_t s_tfs[A3_WARPS][128];
  __shared__ uint32_t s_cur[A3_WARPS][MAXT];
  __shared__ uint32_t s_ord[A3_WARPS][MAXT][128];
  const A3Params& P = PP.A;
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t u = blockIdx.x * A3_WARPS + warp;
  if (u >= P.n_units) return;
  const SegView& S = P.S;
  const AUnit U = P.units[u];
  const uint32_t q = U.q, T = P.q_nterms[q];
  uint32_t* sd = s_docs[warp]; uint32_t* stf = s_tfs[warp]; uint32_t* cur = s_cur[warp];
  if (lane < MAXT) cur[lane] = 0;
  __syncwarp();
  const A3Term tA = a3_load_term(P, q, 0);
  unsigned long long n_blocks = 0, n_hits = 0;
  bool watchdog = false, bad_doc = false;
  for (uint32_t ablk = U.blk_lo; ablk < U.blk_hi; ablk++) {
    uint32_t d[4];
    A3Blk BA; BA.base = nullptr; BA.db = 0; BA.tb = 0; BA.strict = 0;
    uint32_t nA = 128;
    if (ablk < tA.nfull) {
      const uint4 v = a3_decode_docs(P, tA, ablk, lane, BA);
      d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    } else {
      nA = a3_decode_tail(P, tA, sd, stf, lane);
      const uint4 v = ((const uint4*)sd)[lane];
      d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
      __syncwarp();
    }
    n_blocks++;
    uint32_t alive = 0;
#pragma unroll
    for (int b = 0; b < 4; b++) if (lane * 4 + b < nA) {
      if (d[b] < S.max_doc) { alive |= 1u << b; s_ord[warp][0][lane * 4 + b] = ablk * 128u + lane * 4 + b; }
      else bad_doc = true;
    }
    for (uint32_t x = 1; x < T; x++) {
      if (!__any_sync(0xffffffffu, alive != 0)) break;
      const A3Term tX = a3_load_term(P, q, x);
      uint32_t pend = alive;
      for (uint32_t guard = 0;; guard++) {
        if (guard > 130u) { watchdog = true; break; }
        uint32_t m = 0xFFFFFFFFu;
#pragma unroll
        for (int b = 3; b >= 0; b--) if ((pend >> b) & 1u) m = d[b];
#pragma unroll
        for (int o = 16; o; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (m == 0xFFFFFFFFu) break;
        const uint32_t jb = a3_dir_search(S, tX, cur[x], m, lane);
        __syncwarp();
        if (lane == 0) cur[x] = jb;
        uint32_t lastB, lenB; bool x_tail = false;
        A3Blk BX;
        if (jb < tX.nfull) {
          const uint4 v = a3_decode_docs(P, tX, jb, lane, BX);
          __syncwarp();
          ((uint4*)sd)[lane] = v;
          lastB = __shfl_sync(0xffffffffu, v.w, 31); lenB = 128;
          __syncwarp();
        } else {
          x_tail = true; lastB = 0xFFFFFFFFu;
          lenB = (tX.df & 127u) ? a3_decode_tail(P, tX, sd, stf, lane) : 0u;
        }
        n_blocks++;
#pragma unroll
        for (int b = 0; b < 4; b++) {
          if (((pend >> b) & 1u) && d[b] <= lastB) {
            pend &= ~(1u << b);
            bool found = false; uint32_t j = 0;
            if (lenB) { j = lower_bound128(sd, d[b]); found = j < lenB && sd[j] == d[b]; }
            if (!found) alive &= ~(1u << b);
            else s_ord[warp][x][lane * 4 + b] = jb * 128u + j;
          }
        }
        if (x_tail) break;
      }
    }
    const uint32_t cnt = __popc(alive);
    const uint32_t incl = warp_scan_incl(cnt, lane);
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    if (total) {
      unsigned long long base = 0;
      if (lane == 0) base = atomicAdd(PP.c_n, (unsigned long long)total);
      base = __shfl_sync(0xffffffffu, base, 0);
      uint64_t e = base + (incl - cnt);
#pragma unroll
      for (int b = 0; b < 4; b++) if ((alive >> b) & 1u) {
        if (e < PP.c_cap) {
          PP.c_q[e] = q; PP.c_doc[e] = d[b];
          for (uint32_t x = 0; x < T; x++) PP.c_ord[e * MAXT + x] = s_ord[warp][x][lane * 4 + b];
        } else watchdog = true;
        e++;
      }
      n_hits += total;
    }
    __syncwarp();
  }
  if (__any_sync(0xffffffffu, bad_doc)) watchdog = true;
  if (lane == 0) {
    if (n_hits) atomicAdd(PP.counters + 0, n_hits);
    if (n_blocks) atomicAdd(PP.counters + 1, n_blocks);
    if (watchdog) atomicAdd(PP.counters + 2, 1ull);
  }
}

// one warp per candidate (grid-stride over the list): position indexes, the slop-0 phrase count, the score
__global__ void __launch_bounds__(A3_WARPS * 32) k_phrase_match(const PhParams PP) {
  __shared__ float cache[256];
  __shared__ __align__(16) uint32_t s_docs[A3_WARPS][128];
  __shared__ __align__(16) uint32_t s_tfs[A3_WARPS][128];
  __shared__ uint64_t s_pidx[A3_WARPS][MAXT];
  __shared__ uint32_t s_tf[A3_WARPS][MAXT], s_term[A3_WARPS][MAXT], s_ci[A3_WARPS][MAXT], s_base[A3_WARPS][MAXT];
  const A3Params& P = PP.A;
  const SegView& S = P.S;
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (uint32_t i = threadIdx.x; i < 256; i += A3_WARPS * 32) cache[i] = P.cache[i];
  __syncthreads();
  const unsigned long long n = min((unsigned long long)*PP.c_n, (unsigned long long)PP.c_cap);
  bool bad = false;
  for (unsigned long long e = (unsigned long long)blockIdx.x * A3_WARPS + warp; e < n; e += (unsigned long long)gridDim.x * A3_WARPS) {
    const uint32_t q = PP.c_q[e], doc = PP.c_doc[e];
    const uint32_t nd = P.q_nterms[q], L = PP.q_len[q];
    // (1) per distinct term: the posting's tf and position index
    bool ok = true;
    for (uint32_t x = 0; x < nd; x++) {
      const A3Term tx = a3_load_term(P, q, x);
      const uint32_t t = P.q_terms[(size_t)q * MAXT + x];
      const uint32_t ord = PP.c_ord[e * MAXT + x], jb = ord >> 7, kk = ord & 127u;
      uint4 f;
      if (jb < tx.nfull) {
        const uint32_t idx = tx.first + jb, bits = S.b_bits[idx];
        const uint32_t db = bits & 0x3fu, strict = (bits >> 6) & 1u, tb = bits >> 8;
        const uint4* base = P.a128 + tx.adata + (S.b_off[idx] >> 4);
        f = unpack4(base + db, tb, lane);
        f.x += strict; f.y += strict; f.z += strict; f.w += strict;
      } else {
        a3_decode_tail(P, tx, s_docs[warp], s_tfs[warp], lane);
        f = ((const uint4*)s_tfs[warp])[lane];
      }
      const uint32_t s1 = f.x, s2 = s1 + f.y, s3 = s2 + f.z, s4 = s3 + f.w;
      const uint32_t before = warp_scan_incl(s4, lane) - s4;
      const uint32_t sub = kk & 3u;
      const uint32_t my_pre = before + (sub == 0 ? 0u : sub == 1 ? s1 : sub == 2 ? s2 : s3);
      const uint32_t my_tf = sub == 0 ? f.x : sub == 1 ? f.y : sub == 2 ? f.z : f.w;
      const uint32_t pre = __shfl_sync(0xffffffffu, my_pre, kk >> 2), tf = __shfl_sync(0xffffffffu, my_tf, kk >> 2);
      const uint64_t pidx = PP.b_pos[tx.first + jb] + pre;
      if (tf == 0 || pidx + tf > PP.pt_total[t]) ok = false;   // postings and positions disagree: never read past the term
      __syncwarp();
      if (lane == 0) { s_pidx[warp][x] = pidx; s_tf[warp][x] = tf; s_term[warp][x] = t; }
      __syncwarp();
    }
    if (!ok) { bad = true; continue; }
    // (2) the driver: the phrase term with the fewest positions
    uint32_t drv = 0, best = 0xFFFFFFFFu;
    for (uint32_t i = 0; i < L; i++) {
      const uint32_t tf = s_tf[warp][PP.q_slot[(size_t)q * MAXT + i]];
      if (tf < best) { best = tf; drv = i; }
    }
    if (lane < L) { s_ci[warp][lane] = 0; s_base[warp][lane] = PP.q_shift[(size_t)q * MAXT + lane]; }
    __syncwarp();
    const uint32_t dx = PP.q_slot[(size_t)q * MAXT + drv];
    const uint32_t dt = s_term[warp][dx], dtf = s_tf[warp][dx];
    const uint64_t dp = s_pidx[warp][dx];
    uint32_t dbase = PP.q_shift[(size_t)q * MAXT + drv];
    uint32_t count = 0;
    for (uint32_t c0 = 0; c0 < dtf; c0 += 32) {
      const bool valid = c0 + lane < dtf;
      const uint32_t dv = valid ? ph_delta(PP, dt, dp + c0 + lane) : 0u;
      const uint32_t v = dbase + warp_scan_incl(dv, lane);
      dbase = __shfl_sync(0xffffffffu, v, 31);
      bool alive = valid;
      for (uint32_t i = 0; i < L; i++) {
        if (i == drv) continue;
        if (!__any_sync(0xffffffffu, alive)) break;
        const uint32_t xi = PP.q_slot[(size_t)q * MAXT + i];
        const uint32_t ti = s_term[warp][xi], tfi = s_tf[warp][xi];
        const uint64_t pi = s_pidx[warp][xi];
        bool pend = alive;
        for (;;) {
          const uint32_t ci = s_ci[warp][i], cb = s_base[warp][i];
          const uint32_t nc = ci < tfi ? min(32u, tfi - ci) : 0u;
          const uint32_t cv = lane < nc ? ph_delta(PP, ti, pi + ci + lane) : 0u;
          uint32_t c = cb + warp_scan_incl(cv, lane);
          if (lane >= nc) c = 0xFFFFFFFFu;
          const bool last_chunk = ci + 32u >= tfi;
          const uint32_t last = __shfl_sync(0xffffffffu, c, 31);
          uint32_t at = 0;
#pragma unroll
          for (uint32_t step = 16; step; step >>= 1) { const uint32_t pr = __shfl_sync(0xffffffffu, c, at + step - 1u); if (pr < v) at += step; }
          const bool hit = __shfl_sync(0xffffffffu, c, at) == v && at < nc;
          if (pend && (last_chunk || v <= last)) { pend = false; if (!hit) alive = false; }
          if (!__any_sync(0xffffffffu, pend)) break;
          __syncwarp();   // every pending lane is past this chunk: so is every later driver position
          if (lane == 0) { s_ci[warp][i] = ci + 32u; s_base[warp][i] = last; }
          __syncwarp();
        }
      }
      count += __popc(__ballot_sync(0xffffffffu, alive));
    }
    if (count && lane == 0) {
      const float score = a3_term_score(PP.q_weight[q], count, cache[S.fieldnorm[doc]]);
      const uint32_t at = atomicAdd(PP.r_cnt + q, 1u);
      PP.r_key[PP.r_off[q] + at] = ord_f32(score); PP.r_doc[PP.r_off[q] + at] = doc;
    }
    __syncwarp();
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicAdd(PP.counters + 2, 1ull);
}

}  // namespace sb200
