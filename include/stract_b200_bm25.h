/* stract_b200_bm25.h -- C ABI of hot path 2: BM25 posting-list scoring + top-k collection over
 * tantivy-format posting lists (part of libstract_b200.so; conventions as in stract_b200.h).
 *
 * Replaces, per segment (paths relative to /root/reference/crates):
 *   (A) tantivy-native top-k:  TopDocs::collect_segment -> Weight::for_each_pruning -> Intersection /
 *       block_wand -> TermScorer::score -> TopNComputer
 *         tantivy/src/collector/top_score_collector.rs:385-413,501-564, tantivy/src/query/weight.rs:47-60,
 *         tantivy/src/query/intersection.rs:14-160, tantivy/src/query/boolean_query/block_wand.rs:148-214,
 *         tantivy/src/query/term_query/term_scorer.rs:119-123, tantivy/src/query/bm25.rs:182-196
 *   (B) Stract's recall stage: TweakedScoreTopCollector + InitialSegmentScoreTweaker::score
 *       (Sum coefficient x signal in f64) with TextFieldData::bm25 re-seeking its own cursors
 *         core/src/collector/top_docs.rs:404-490, core/src/ranking/initial.rs:79-93,
 *         core/src/ranking/computer/mod.rs:109-124, core/src/ranking/bm25.rs:97-102,136-150
 * The posting bytes are consumed exactly as tantivy writes them (128-doc BitPacker4x blocks, strict
 * deltas, tf-1, VInt tail, skip entries: tantivy/src/postings/{serializer.rs:365-462,skip.rs:186-238}).
 *
 * The GPU scores exhaustively (every posting of every query term) and returns the exact top-k under the
 * reference's total order (score descending, then doc ascending; tantivy/src/collector/top_collector.rs:50-66).
 * Pruning in the reference (Block-WAND, TopNComputer threshold) only drops documents that cannot enter the
 * top-k, so results are identical.  f32/f64 expressions are evaluated in the reference's operation order
 * without FMA contraction; see DESIGN.md for the one documented deviation (the association of the f32 sum
 * in tantivy OR queries with >= 3 terms, which in the reference depends on the pruning history).
 */
#ifndef STRACT_B200_BM25_H
#define STRACT_B200_BM25_H
#include "stract_b200.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct sb200_segment sb200_segment;
typedef struct sb200_signals sb200_signals;

/* TermInfo{doc_freq, postings_range} of one term, tantivy/src/postings/term_info.rs:9-14 */
typedef struct { uint64_t postings_off; uint64_t postings_len; uint32_t doc_freq; uint32_t _pad; } sb200_term_info;

#define SB200_RECORD_BASIC 0            /* IndexRecordOption::Basic: 5-byte skip entries, no tf */
#define SB200_RECORD_FREQS 1            /* WithFreqs: 8-byte skip entries */
#define SB200_RECORD_FREQS_POSITIONS 2  /* WithFreqsAndPositions: 12-byte skip entries */

/* Opens one field of one segment (InvertedIndexReader + FieldNormReader, tantivy/src/index/
 * inverted_index_reader.rs:66-68, tantivy/src/fieldnorm/reader.rs:128-136): copies the postings file and the
 * 1-byte-per-doc fieldnorm ids into HBM and builds a per-block directory (last doc, byte offset, bit widths)
 * from the skip lists so blocks are randomly addressable on the device.  Terms are addressed by their ordinal
 * in `terms` afterwards. */
SB200_API int sb200_segment_create(const uint8_t* postings_file, uint64_t postings_len, const sb200_term_info* terms,
                                   uint32_t n_terms, const uint8_t* fieldnorm_ids, uint32_t max_doc,
                                   int record_option, int device, sb200_segment** out);
SB200_API void sb200_segment_destroy(sb200_segment* seg);

/* The "term ordinal -> TermInfo" half of the term dictionary (SURVEY 8(f) rank 2): decodes a whole tantivy TermInfoStore
 * (tantivy/src/termdict/fst_termdict/term_info_store.rs: 256-term blocks, a 47-byte TermInfoBlockMeta each, bit-packed
 * offsets) on the device, one thread per ordinal, into the array sb200_segment_create takes.  `store` may be host or
 * device memory, `infos` receives min(cap, n) entries, *n_terms the number of terms.  (The FST that maps term bytes to an
 * ordinal is an external crate that is not part of the reference tree; callers address terms by ordinal.) */
SB200_API int sb200_term_info_store_decode(const uint8_t* store, uint64_t len, int device, sb200_term_info* infos, uint64_t cap,
                                           uint64_t* n_terms);

/* The positions half of the same store: positions_range [start, end) of every term, the end being the next term's start
 * (term_info_store.rs:66-91), min(cap, n) entries; what sb200_segment_attach_positions takes. */
SB200_API int sb200_term_info_store_decode_positions(const uint8_t* store, uint64_t len, int device, uint64_t* pos_start, uint64_t* pos_end,
                                                     uint64_t cap, uint64_t* n_terms);

typedef struct { uint64_t n_terms, n_blocks, n_postings, hbm_bytes; uint32_t max_doc; uint32_t _pad; double stage_ms; } sb200_segment_info;

/* Attaches the field's positions file (tantivy/src/positions/mod.rs:7-30: per term VInt(#blocks), one bit width per block,
 * 128-delta BitPacker4x blocks, a vint tail of the remaining deltas) to a WithFreqsAndPositions segment (record option 2,
 * else SB200_EINVAL); term t's bytes are [pos_start[t], pos_end[t]).  The file goes to HBM with a per-128-position block
 * directory, a 16-byte aligned copy of the bitpacked blocks and, per posting block, the index of its first position (the
 * skip entries' tf sums, what SkipReader::position_offset accumulates, tantivy/src/postings/skip.rs:244-266).  Every term is
 * validated first (range inside the file, block count == its term frequency sum / 128, widths <= 32, blocks inside the range,
 * exactly sum % 128 tail vints): SB200_EFORMAT and nothing attached otherwise.  sb200_segment_get_info().hbm_bytes counts it. */
SB200_API int sb200_segment_attach_positions(sb200_segment* seg, const uint8_t* positions_file, uint64_t len, const uint64_t* pos_start,
                                             const uint64_t* pos_end);
SB200_API int sb200_segment_get_info(const sb200_segment* seg, sb200_segment_info* info);

/* Row-major table of per-document numeric signal scores in HBM ([max_doc][n_cols] f64): what the numeric
 * CoreSignals read per candidate (core/src/ranking/signals/core/non_text.rs).  Column j holds the signal's
 * *score* (the host applies value->score transforms such as score_rank once at open time). */
SB200_API int sb200_signals_create(const double* const* columns, uint32_t n_cols, uint32_t max_doc, int device, sb200_signals** out);
/* The same table built from the RAW fast-field columns: the library applies the numeric CoreSignals' value -> score
 * transforms (core/src/ranking/signals/core/non_text.rs) on the device, one pass per column at open time.
 *   kind                   reference                                            raw column
 *   SB200_NUM_IDENTITY     HostCentrality, PageCentrality (:117-155, :203-241)  f64
 *   SB200_NUM_RANK         score_rank (:50-59): HostCentralityRank, PageCentralityRank   u64  (evaluated on the host: libm ln)
 *   SB200_NUM_BOOL         IsHomepage (:289-332)                                bool8
 *   SB200_NUM_BOOL_NOT     HasAds: score = !likely_has_ads (:730-771)           bool8
 *   SB200_NUM_INVERSE      score_trackers / score_digits / score_slashes (:61-74): TrackerScore, UrlDigits, UrlSlashes   u64
 *   SB200_NUM_FETCH_TIME   FetchTimeMs over fetch_time_ms_cache (1000 entries, computer/mod.rs:257-259)                  u64
 *   SB200_NUM_UPDATE_TIME  UpdateTimestamp: score_timestamp (:25-42) over update_time_cache; p0 = current_timestamp      u64
 *   SB200_NUM_LINK_DENSITY score_link_density (:76-83)                          f64
 *   SB200_NUM_REGION       score_region (:85-101): lut[region id] = RegionCount::score (count / total, webpage/region.rs:219-227),
 *                          p1 != 0: a region other than All is selected, p0 = its id (+50); lut NULL = no RegionCount: all 0     u64 */
#define SB200_NUM_IDENTITY 0u
#define SB200_NUM_RANK 1u
#define SB200_NUM_BOOL 2u
#define SB200_NUM_BOOL_NOT 3u
#define SB200_NUM_INVERSE 4u
#define SB200_NUM_FETCH_TIME 5u
#define SB200_NUM_UPDATE_TIME 6u
#define SB200_NUM_LINK_DENSITY 7u
#define SB200_NUM_REGION 8u
#define SB200_NUM_U64 0u
#define SB200_NUM_F64 1u
#define SB200_NUM_BOOL8 2u
typedef struct {
  uint32_t kind, dtype;      /* SB200_NUM_* transform, SB200_NUM_U64 / F64 / BOOL8 element type of `raw` */
  const void* raw;           /* [max_doc], host or device */
  double p0, p1;
  const double* lut; uint32_t lut_len, _pad;
} sb200_numeric_column;
SB200_API int sb200_signals_create_raw(const sb200_numeric_column* cols, uint32_t n_cols, uint32_t max_doc, int device, sb200_signals** out);
/* rows [first_doc, first_doc + n_docs) of the table, row-major [n_docs][n_cols] (inspection / tests) */
SB200_API int sb200_signals_read(const sb200_signals* s, uint32_t first_doc, uint32_t n_docs, double* rows_out);
SB200_API void sb200_signals_destroy(sb200_signals* s);

#define SB200_MODE_AND 0     /* all clauses Occur::Must  -> Intersection, score = left + right + sum(others) */
#define SB200_MODE_OR 1      /* all clauses Occur::Should -> union, score = f32 sum over matching terms in query order */
#define SB200_MODE_OR_WAND 2 /* the same union with tantivy's Block-Max WAND replayed step by step (block_wand.rs:148-214): the f32
                               sum of a document's term scores then has the association the reference's pruning history gives it,
                               so scores and doc order match the reference bit for bit for ANY number of terms.  10-100x slower
                               than SB200_MODE_OR, whose sums are in query order (identical for <= 2 terms). */
#define SB200_NO_TERM 0xFFFFFFFFu  /* padding for queries shorter than the batch arity */
#define SB200_MAX_QUERY_TERMS 8
#define SB200_MAX_K 4096

/* A batch of same-arity queries over one field.  Weights come from the host exactly as the reference computes
 * them: `weight[q][t]` = Bm25Weight.weight (idf*(1+K1), tantivy/src/query/bm25.rs:161-162) for path A or the
 * Stract idf (core/src/ranking/bm25.rs:124-134) for path B; `tf_cache256` = the field's 256-entry
 * K1*(1-B+B*fieldnorm/avg) table (bm25.rs:58-68), shared by every term of the field. */
typedef struct {
  uint32_t n_queries, n_terms;
  const uint32_t* term_ords;   /* [n_queries*n_terms], SB200_NO_TERM to pad */
  const float* weights;        /* [n_queries*n_terms] */
  const float* tf_cache256;    /* [256] */
  int mode;                    /* SB200_MODE_AND / SB200_MODE_OR */
  uint32_t k;                  /* TopDocs::with_limit(k) */
} sb200_bm25_batch;

/* ms: device time of the whole call on the handle's stream (query H2D + kernel + result D2H);
 * kernel_ms: the k_topk launch alone (CUDA events around it). */
typedef struct { uint64_t postings_scored; uint64_t docs_scored; uint64_t blocks_decoded; float ms; float kernel_ms; } sb200_bm25_stats;

/* Path A.  Outputs are host (or device) arrays: docs/scores [n_queries*k] in rank order (score desc, doc asc),
 * n_out[q] <= k entries valid per query. */
SB200_API int sb200_bm25_topk_batch(sb200_segment* seg, const sb200_bm25_batch* batch, uint32_t* docs, float* scores,
                                    uint32_t* n_out, sb200_bm25_stats* stats);
/* single query convenience (a batch of one) */
SB200_API int sb200_bm25_topk(sb200_segment* seg, const uint32_t* term_ords, const float* weights, uint32_t n_terms,
                              const float* tf_cache256, int mode, uint32_t k, uint32_t* docs, float* scores, uint32_t* n_out);

/* Path B.  Candidates = union of the query terms' postings (MainCollector does not require scoring, the docset
 * is the Should-union), per candidate
 *   total = coeff_text * (bm25 as f64) + sum_j coeffs[j] * signals[doc][j]        (f64, that order)
 *   bm25  = f32 sum over the query terms in query order of idf*((tf*(k1+1))/(tf+cache[fieldnorm_id])), tf=0 -> 0
 * top-k by (total desc, doc asc).  max_docs > 0 stops after that many candidates in ascending doc order
 * (ShortCircuitQuery, tantivy/src/query/shortcircuit.rs:100-133). */
typedef struct {
  sb200_bm25_batch q;          /* mode ignored (always the union); weights = Stract idf */
  float k1;                    /* Bm25Constants.k1 of the field (1.2) */
  double coeff_text;           /* coefficient of the field's BM25 signal */
  const sb200_signals* signals;/* nullable */
  const double* coeffs;        /* [signals.n_cols] */
  uint32_t max_docs; uint32_t _pad;
} sb200_signal_batch;
SB200_API int sb200_signal_topk_batch(sb200_segment* seg, const sb200_signal_batch* batch, uint32_t* docs, double* totals,
                                      uint32_t* n_out, sb200_bm25_stats* stats);

/* Path B over SEVERAL text fields of one segment (SURVEY 8(f) rank 3): the recall-stage signal set of
 * SignalComputeOrder::compute (core/src/ranking/computer/order.rs:17-135) evaluated per candidate exactly as
 * InitialSegmentScoreTweaker::score sums it (core/src/ranking/initial.rs:79-93):
 *     total = sum over the ops, in the order given, of coeff * score            (f64)
 * A field is one sb200_segment (the same tantivy segment opened per field: equal max_doc).  A query gives every field
 * its terms as SLOTS in query order -- slot_field[q][x] = field index (0xFF pads), slot_term = the term's ordinal in that
 * field's segment or SB200_NO_TERM when the segment does not hold it (SegmentPostings::empty(): the slot still counts in
 * num_query_terms), slot_idf = MultiBm25Weight's idf (core/src/ranking/bm25.rs:52-92), slot_idf_f = MultiBm25FWeight's
 * (doc_freq of the AllBody field, core/src/ranking/bm25f.rs:40-45,88-131).  Op kinds (computer/mod.rs:66-163):
 *   SB200_OP_BM25      TextFieldData::bm25 of `field`      f32 sum over its slots of idf*((tf*(k1+1))/(tf+cache[id])), tf=0 -> 0
 *   SB200_OP_BM25F     Bm25F: f64 sum over the fields (in field order) of TextFieldData::bm25f -- the same saturation
 *                      with slot_idf_f and tf scaled by the field's bm25f_coefficient as f32 (bm25f.rs:167-180)
 *   SB200_OP_COVERAGE  matching slots / num_query_terms of `field` (f64)
 *   SB200_OP_IDF_SUM   f32 sum of slot_idf over the matching slots of `field`
 *   SB200_OP_NUMERIC   column `col` of the signal table
 * chain != 0 marks the members of an n-gram group in the reference's order (largest n first; 1 = first member):
 * score *= 0.4^hits and hits += (score > 0) (NGRAM_DAMPENING, computer/order.rs:95-135).
 * Optic rule boosts (SignalComputer::boosts, computer/mod.rs:471-497): a rule whose docset is one posting list is a slot
 * with slot_field = field | 0x80 and its boost in slot_boost (negative = downrank); rule slots are probed for the documents
 * being scored and never produce candidates; total *= (downrank > boost ? 1/(1 + downrank - boost) : boost - downrank + 1)
 * with the f64 sums taken in slot order.  slot_boost may be NULL when no slot is a rule.
 * Candidates are the union of the TEXT slots' postings; top-k by (total desc, doc asc).  Limits: <= 6 fields, <= 16 slots
 * per query, <= 32 ops. */
#define SB200_OP_BM25 0u
#define SB200_OP_BM25F 1u
#define SB200_OP_COVERAGE 2u
#define SB200_OP_IDF_SUM 3u
#define SB200_OP_NUMERIC 4u
typedef struct { sb200_segment* seg; const float* tf_cache256; float k1; float bm25f_coefficient; } sb200_signal_field;
typedef struct { uint32_t kind, field, chain, col; double coeff; } sb200_signal_op;
typedef struct {
  uint32_t n_queries, n_slots;        /* slots per query (row width of the four arrays below) */
  const uint8_t* slot_field;          /* [n_queries*n_slots] */
  const uint32_t* slot_term;          /* [n_queries*n_slots] */
  const float* slot_idf;              /* [n_queries*n_slots] */
  const float* slot_idf_f;            /* [n_queries*n_slots] */
  uint32_t n_fields, n_ops;
  const sb200_signal_field* fields;   /* [n_fields], in TextFieldEnum order */
  const sb200_signal_op* ops;         /* [n_ops], in SignalComputeOrder order */
  const sb200_signals* signals;       /* nullable unless an op is SB200_OP_NUMERIC */
  uint32_t k, _pad;
  const double* slot_boost;           /* [n_queries*n_slots], read for rule slots only; nullable */
} sb200_multi_signal_batch;
SB200_API int sb200_multi_signal_topk_batch(const sb200_multi_signal_batch* batch, uint32_t* docs, double* totals, uint32_t* n_out,
                                            sb200_bm25_stats* stats);

/* Phrase queries with slop 0: tantivy PhraseQuery::new / new_with_offset (query/phrase_query/phrase_query.rs:35-53) collected by
 * TopDocs on one segment.  Per query the phrase terms term_ords[q][0..lens[q]) with their offsets (any order: the phrase
 * count does not depend on it); a document matches when every term occurs at (start + offset), PhraseScorer's count is the
 * number of such starts (phrase_scorer.rs:435-505 with slop 0) and the score is weights[q] * (count / (count +
 * tf_cache256[fieldnorm id])) (PhraseScorer::score, phrase_scorer.rs:540-549; Bm25Weight::score, bm25.rs:182-196).
 * weights[q] = Bm25Weight::for_terms(..).weight: (1 + K1) times the f32 idf sum over the terms in offset order
 * (bm25.rs:98-134), times the boost.  A query with an SB200_NO_TERM among its terms matches nothing (PhraseWeight::phrase_scorer
 * returns None, phrase_weight.rs:53-62); lens[q] < 2 (phrase_query.rs:49-52) or a segment without positions
 * (phrase_query.rs:106-118) is SB200_EINVAL.  Outputs as sb200_bm25_topk_batch; stats: postings_scored = sum of the phrase
 * terms' doc_freq, docs_scored = documents containing every term (the ones whose positions were matched). */
typedef struct {
  uint32_t n_queries, n_terms;   /* n_terms = row width, 2 <= n_terms <= SB200_MAX_QUERY_TERMS */
  const uint32_t* term_ords;     /* [n_queries*n_terms]; SB200_NO_TERM = term absent from this segment */
  const uint32_t* offsets;       /* [n_queries*n_terms]: PhraseQuery::new_with_offset positions */
  const uint8_t* lens;           /* [n_queries]: phrase length, 2..n_terms */
  const float* weights;          /* [n_queries] */
  const float* tf_cache256;      /* [256] */
  uint32_t k;
} sb200_phrase_batch;
SB200_API int sb200_phrase_topk_batch(sb200_segment* seg, const sb200_phrase_batch* batch, uint32_t* docs, float* scores,
                                      uint32_t* n_out, sb200_bm25_stats* stats);

/* Host-side writer of tantivy-format posting lists (PostingsSerializer for IndexRecordOption::WithFreqs,
 * tantivy/src/postings/serializer.rs:343-462), used to build synthetic / test segments.  Terms are given
 * CSR-style: term t owns docs[term_off[t]..term_off[t+1]) (ascending) and the matching tfs (>= 1).
 * Call with out == NULL to get the byte size. */
SB200_API int sb200_postings_encode(const uint32_t* docs, const uint32_t* tfs, const uint64_t* term_off, uint32_t n_terms,
                                    const uint8_t* fieldnorm_ids, uint32_t max_doc, float avg_fieldnorm, uint8_t* out,
                                    uint64_t out_cap, uint64_t* out_len, sb200_term_info* infos, int threads);
/* The same writer with the record option spelled out: 1 = WithFreqs (8-byte skip entries), 2 = WithFreqsAndPositions,
 * what Stract's position-bearing text fields use (core/src/schema/text_field.rs:124-130): 12-byte skip entries that carry
 * the block's term-frequency sum (tantivy/src/postings/skip.rs:52-76,217-232); the positions themselves are another file. */
SB200_API int sb200_postings_encode_ex(const uint32_t* docs, const uint32_t* tfs, const uint64_t* term_off, uint32_t n_terms,
                                       const uint8_t* fieldnorm_ids, uint32_t max_doc, float avg_fieldnorm, int record_option,
                                       uint8_t* out, uint64_t out_cap, uint64_t* out_len, sb200_term_info* infos, int threads);
/* Host-side writer of the positions file (PositionSerializer, tantivy/src/positions/serializer.rs) for the same CSR: `positions`
 * holds sum(tfs) entries, every posting's absolute positions (strictly ascending within the document), posting after posting;
 * a document's deltas restart from 0 (postings/serializer.rs:191-205).  Term t's bytes go to [pos_start[t], pos_end[t])
 * (both nullable).  Call with out == NULL to get the byte size. */
SB200_API int sb200_positions_encode(const uint32_t* docs, const uint32_t* tfs, const uint64_t* term_off, uint32_t n_terms,
                                     const uint32_t* positions, uint8_t* out, uint64_t out_cap, uint64_t* out_len, uint64_t* pos_start,
                                     uint64_t* pos_end, int threads);
/* idf(doc_freq, doc_count) = ln(1 + (N - n + 0.5) / (n + 0.5)) in f32 (tantivy/src/query/bm25.rs:52-56,
 * core/src/ranking/bm25.rs:23-27) for an array of doc_freqs; tantivy_weight != 0 returns Bm25Weight.weight = idf * (1 + K1). */
SB200_API int sb200_bm25_idf(const uint32_t* doc_freq, uint64_t n, uint64_t doc_count, int tantivy_weight, float* out);
/* FIELD_NORMS_TABLE (tantivy/src/fieldnorm/code.rs:13-270) as the closed-form byte code it is tested against */
SB200_API uint32_t sb200_fieldnorm_id_to_value(uint8_t id);
SB200_API uint8_t sb200_fieldnorm_value_to_id(uint32_t fieldnorm);

#ifdef __cplusplus
}
#endif
#endif
