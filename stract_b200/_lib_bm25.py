"""ctypes prototypes of the path-2 (BM25) entry points (include/stract_b200_bm25.h)."""
import ctypes as C


class TermInfo(C.Structure):
    _fields_ = [("postings_off", C.c_uint64), ("postings_len", C.c_uint64), ("doc_freq", C.c_uint32), ("_pad", C.c_uint32)]


class SegmentInfo(C.Structure):
    _fields_ = [("n_terms", C.c_uint64), ("n_blocks", C.c_uint64), ("n_postings", C.c_uint64), ("hbm_bytes", C.c_uint64),
                ("max_doc", C.c_uint32), ("_pad", C.c_uint32), ("stage_ms", C.c_double)]


class Bm25Batch(C.Structure):
    _fields_ = [("n_queries", C.c_uint32), ("n_terms", C.c_uint32), ("term_ords", C.c_void_p), ("weights", C.c_void_p),
                ("tf_cache256", C.c_void_p), ("mode", C.c_int), ("k", C.c_uint32)]


class Bm25Stats(C.Structure):
    _fields_ = [("postings_scored", C.c_uint64), ("docs_scored", C.c_uint64), ("blocks_decoded", C.c_uint64),
                ("ms", C.c_float), ("kernel_ms", C.c_float)]


class SignalBatch(C.Structure):
    _fields_ = [("q", Bm25Batch), ("k1", C.c_float), ("coeff_text", C.c_double), ("signals", C.c_void_p),
                ("coeffs", C.c_void_p), ("max_docs", C.c_uint32), ("_pad", C.c_uint32)]


class SignalField(C.Structure):
    _fields_ = [("seg", C.c_void_p), ("tf_cache256", C.c_void_p), ("k1", C.c_float), ("bm25f_coefficient", C.c_float)]


class NumericColumn(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("dtype", C.c_uint32), ("raw", C.c_void_p), ("p0", C.c_double), ("p1", C.c_double),
                ("lut", C.c_void_p), ("lut_len", C.c_uint32), ("_pad", C.c_uint32)]


class SignalOp(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("field", C.c_uint32), ("chain", C.c_uint32), ("col", C.c_uint32), ("coeff", C.c_double)]


class MultiSignalBatch(C.Structure):
    _fields_ = [("n_queries", C.c_uint32), ("n_slots", C.c_uint32), ("slot_field", C.c_void_p), ("slot_term", C.c_void_p),
                ("slot_idf", C.c_void_p), ("slot_idf_f", C.c_void_p), ("n_fields", C.c_uint32), ("n_ops", C.c_uint32),
                ("fields", C.c_void_p), ("ops", C.c_void_p), ("signals", C.c_void_p), ("k", C.c_uint32), ("_pad", C.c_uint32),
                ("slot_boost", C.c_void_p)]


class PhraseBatch(C.Structure):
    _fields_ = [("n_queries", C.c_uint32), ("n_terms", C.c_uint32), ("term_ords", C.c_void_p), ("offsets", C.c_void_p),
                ("lens", C.c_void_p), ("weights", C.c_void_p), ("tf_cache256", C.c_void_p), ("k", C.c_uint32)]


def proto(L, f):
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    f("sb200_segment_create", i32, vp, u64, vp, u32, vp, u32, i32, i32, C.POINTER(vp))
    f("sb200_segment_destroy", None, vp)
    f("sb200_segment_get_info", i32, vp, C.POINTER(SegmentInfo))
    f("sb200_signals_create", i32, vp, u32, u32, i32, C.POINTER(vp))
    f("sb200_signals_create_raw", i32, vp, u32, u32, i32, C.POINTER(vp))
    f("sb200_signals_read", i32, vp, u32, u32, vp)
    f("sb200_signals_destroy", None, vp)
    f("sb200_bm25_topk_batch", i32, vp, C.POINTER(Bm25Batch), vp, vp, vp, C.POINTER(Bm25Stats))
    f("sb200_bm25_topk", i32, vp, vp, vp, u32, vp, i32, u32, vp, vp, vp)
    f("sb200_signal_topk_batch", i32, vp, C.POINTER(SignalBatch), vp, vp, vp, C.POINTER(Bm25Stats))
    f("sb200_multi_signal_topk_batch", i32, C.POINTER(MultiSignalBatch), vp, vp, vp, C.POINTER(Bm25Stats))
    f("sb200_postings_encode", i32, vp, vp, vp, u32, vp, u32, C.c_float, vp, u64, C.POINTER(u64), vp, i32)
    f("sb200_term_info_store_decode", i32, vp, u64, i32, vp, u64, C.POINTER(u64))
    f("sb200_postings_encode_ex", i32, vp, vp, vp, u32, vp, u32, C.c_float, i32, vp, u64, C.POINTER(u64), vp, i32)
    f("sb200_bm25_idf", i32, vp, u64, u64, i32, vp)
    f("sb200_fieldnorm_id_to_value", u32, C.c_uint8)
    f("sb200_fieldnorm_value_to_id", C.c_uint8, u32)
    f("sb200_term_info_store_decode_positions", i32, vp, u64, i32, vp, vp, u64, C.POINTER(u64))
    f("sb200_segment_attach_positions", i32, vp, vp, u64, vp, vp)
    f("sb200_phrase_topk_batch", i32, vp, C.POINTER(PhraseBatch), vp, vp, vp, C.POINTER(Bm25Stats))
    f("sb200_positions_encode", i32, vp, vp, vp, u32, vp, vp, u64, C.POINTER(u64), vp, vp, i32)
