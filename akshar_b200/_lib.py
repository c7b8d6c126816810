"""ctypes binding of libakshar_b200.so (C ABI in include/akshar_b200.h).

There is no CPU fallback: if the CUDA library has not been built (``python -c "import __graft_entry__ as g; g.build()"``)
or no B200 is present, importing/using the batch path raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('AKSHAR_B200_LIB') or os.path.join(_HERE, 'lib', 'libakshar_b200.so')

OK, E_ARG, E_CUDA, E_MODEL, E_NOMODEL, E_WORKSPACE = 0, -1, -2, -3, -4, -5
ST_OVERFLOW, ST_NFC_SEGMENT, ST_PATHOLOGICAL, ST_ALPHABET, ST_SPIN, ST_WORD, ST_INTERNAL, ST_BAD_ID = 1, 2, 4, 8, 16, 32, 64, 128
ST_TEMPLATE, ST_PAIR_TRUNC, ST_PACK_LONG = 256, 512, 1024
NORM_ROMAN, NORM_FILTER, NORM_COLLAPSE, NORM_CLEAN, NORM_NO_NFC = 1, 2, 4, 6, 8
SEG_CLUSTERS, SEG_MATRAS, SEG_RUNS, SEG_MASK = 1, 2, 4, 8
MODE_TILES, MODE_ROWS = 0, 1
OUT_IDS_U16, OUT_SPLITS_I32 = 1, 2
WORDS_HINDI, WORDS_SPLIT = 0, 1
FORM_DECODE, FORM_DETOKENIZE = 0, 1
MERGE_AKSHARA, MERGE_NUKTA = 0, 1
WIN_TRUNCATE, WIN_OVERFLOW, WIN_TRUNC_LEFT, WIN_PAD_LEFT, WIN_ONLY_FIRST, WIN_ONLY_SECOND = 1, 2, 4, 8, 16, 32
TIMERS = {'ak_nf3_classify_kernel': 0, 'ak_nf_write_kernel': 1, 'ak_resolve_kernel<bpe>': 2, 'ak_seg_off_kernel<emit>': 3, 'ak_seg_mask_kernel': 3,
          'ak_resolve_kernel<unigram>': 4, 'ak_words_kernel': 5, 'ak_emit_kernel': 6, 'ak_wtok_kernel': 7, 'ak_dec_kernel': 8, 'ak_lines_kernel': 9}

SYMBOLS = (
    'akshar_version', 'akshar_status_str', 'akshar_ctx_create', 'akshar_ctx_destroy', 'akshar_last_error',
    'akshar_workspace_bytes', 'akshar_normalize_batch', 'akshar_segment_batch', 'akshar_signature_batch',
    'akshar_load_bpe_json', 'akshar_load_spm_model', 'akshar_vocab_size', 'akshar_vocab_token',
    'akshar_encode_bpe_batch', 'akshar_encode_unigram_batch', 'akshar_tokenizer_encode_batch', 'akshar_tokenizer_encode_batch_ex',
    'akshar_launch_count', 'akshar_timing_enable', 'akshar_timing_read', 'akshar_word_cache_hold', 'akshar_word_cache_stats', 'akshar_word_tokenize_batch', 'akshar_decode_workspace_bytes', 'akshar_decode_batch', 'akshar_composition_batch', 'akshar_merge_workspace_bytes', 'akshar_merge_clusters_batch', 'akshar_lines_workspace_bytes', 'akshar_lines_batch', 'akshar_join_rows', 'akshar_normalize_segment_batch',
    'akshar_windows_workspace_bytes', 'akshar_windows_count', 'akshar_windows_write', 'akshar_pair_windows_count',
    'akshar_pair_windows_write', 'akshar_pack_workspace_bytes', 'akshar_pack_count', 'akshar_pack_write', 'akshar_mlm_mask',
)

_lib = None


class AksharCudaError(RuntimeError):
    pass


def load():
    """dlopen the library and declare every prototype; raises if it has not been built"""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AksharCudaError(
            'akshar_b200: %s is missing -- build it with `python -c "import __graft_entry__ as g; g.build()"`; '
            'there is no CPU fallback for the batch path' % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    c = ctypes
    vp, i64, i32, u32, sz = c.c_void_p, c.c_int64, c.c_int, c.c_uint32, c.c_size_t
    L.akshar_version.restype = i32
    L.akshar_status_str.restype = c.c_char_p
    L.akshar_status_str.argtypes = [i32]
    L.akshar_ctx_create.argtypes = [i32, c.POINTER(vp)]
    L.akshar_ctx_destroy.argtypes = [vp]
    L.akshar_ctx_destroy.restype = None
    L.akshar_last_error.argtypes = [vp]
    L.akshar_last_error.restype = c.c_char_p
    L.akshar_workspace_bytes.argtypes = [i64, i64]
    L.akshar_workspace_bytes.restype = sz
    L.akshar_normalize_batch.argtypes = [vp, vp, vp, i64, i64, i64, u32, i32, vp, i64, vp, vp, vp, sz, vp]
    L.akshar_segment_batch.argtypes = [vp, vp, vp, i64, i64, i64, u32, i32, vp, i64, vp, vp, vp, i64, vp, vp, vp, sz, vp]
    L.akshar_signature_batch.argtypes = [vp, vp, vp, i64, i64, i64, vp, i64, vp, vp, vp, sz, vp]
    L.akshar_word_tokenize_batch.argtypes = [vp, vp, vp, i64, i64, i64, i32, vp, vp, i64, vp, vp, vp, vp, sz, vp]
    L.akshar_decode_workspace_bytes.argtypes = [i64, i64]
    L.akshar_decode_workspace_bytes.restype = sz
    L.akshar_decode_batch.argtypes = [vp, i32, i32, vp, i32, i64, vp, i64, vp, i64, vp, vp, vp, sz, vp]
    L.akshar_composition_batch.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp, vp, vp]
    L.akshar_merge_workspace_bytes.argtypes = [i64]
    L.akshar_merge_workspace_bytes.restype = sz
    L.akshar_merge_clusters_batch.argtypes = [vp, vp, vp, i64, vp, vp, i64, i32, vp, i64, vp, vp, vp, sz, vp]
    L.akshar_lines_workspace_bytes.argtypes = [i64, i64]
    L.akshar_lines_workspace_bytes.restype = sz
    L.akshar_lines_batch.argtypes = [vp, vp, i64, vp, i64, vp, i64, vp, vp, sz, vp]
    L.akshar_join_rows.argtypes = [vp, vp, vp, i64, i32, vp, vp]
    L.akshar_normalize_segment_batch.argtypes = [vp, vp, vp, i64, i64, i64, u32, u32, vp, i64, vp, vp, vp, vp, i64, vp, vp, sz, vp]
    L.akshar_windows_workspace_bytes.argtypes = [i64]
    L.akshar_windows_workspace_bytes.restype = sz
    L.akshar_windows_count.argtypes = [vp, i32, vp, i32, vp, i64, i64, i64, u32, vp, vp, vp, sz, vp]
    L.akshar_windows_write.argtypes = [vp, i32, vp, i32, vp, vp, i64, i64, i64, i64, u32, i64, i64, vp, vp, vp, vp]
    L.akshar_pair_windows_count.argtypes = [vp, i32, vp, vp, vp, vp, i32, i64, i64, i64, u32, vp, vp, vp, sz, vp]
    L.akshar_pair_windows_write.argtypes = [vp, i32, vp, vp, vp, vp, i32, vp, i64, i64, i64, i64, u32, i64, i64, vp, vp, vp, vp]
    L.akshar_pack_workspace_bytes.argtypes = [i64]
    L.akshar_pack_workspace_bytes.restype = sz
    L.akshar_pack_count.argtypes = [vp, vp, i32, vp, i64, vp, vp, i64, i64, i64, vp, vp, sz, vp]
    L.akshar_pack_write.argtypes = [vp, vp, i32, vp, i64, vp, vp, i64, i64, i64, i64, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp,
                                    sz, vp]
    L.akshar_mlm_mask.argtypes = [vp, i32, vp, i64, i64, c.c_uint64, u32, c.c_uint64, c.POINTER(c.c_uint64), i64, i64, vp, vp]
    L.akshar_load_bpe_json.argtypes = [vp, c.c_char_p, sz]
    L.akshar_load_spm_model.argtypes = [vp, c.c_char_p, sz]
    L.akshar_vocab_size.argtypes = [vp, i32]
    L.akshar_vocab_token.argtypes = [vp, i32, i32, c.POINTER(vp), c.POINTER(i32), c.POINTER(i32)]
    L.akshar_encode_bpe_batch.argtypes = [vp, vp, vp, i64, i64, i64, i32, vp, i64, vp, vp, vp, sz, vp]
    L.akshar_encode_unigram_batch.argtypes = [vp, vp, vp, i64, i64, i64, i32, vp, i64, vp, vp, vp, sz, vp]
    L.akshar_tokenizer_encode_batch.argtypes = [vp, vp, vp, i64, i64, i64, u32, i32, i32, vp, i64, vp, vp, i64, vp, vp, vp, sz, vp]
    L.akshar_tokenizer_encode_batch_ex.argtypes = [vp, vp, vp, i64, i64, i64, u32, i32, i32, vp, i64, vp, vp, i64, vp, u32, vp, vp, sz, vp]
    L.akshar_timing_enable.argtypes = [vp, i32]
    L.akshar_word_cache_hold.argtypes = [vp, i32]
    L.akshar_word_cache_stats.argtypes = [vp, i32, vp, vp]
    L.akshar_timing_read.argtypes = [vp, i32, c.POINTER(c.c_float)]
    L.akshar_launch_count.argtypes = [vp]
    L.akshar_launch_count.restype = i64
    _lib = L
    return L
