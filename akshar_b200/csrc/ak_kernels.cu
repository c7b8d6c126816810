// libakshar_b200.so -- CUDA kernels (sm_100a) + the C ABI declared in include/akshar_b200.h.
//
// Every batch kernel is persistent (gridDim = SMs x resident CTAs); a CTA draws tile numbers from an atomic
// ticket, each thread walks one byte span of the tile (ak_text_core.cuh / ak_subword.cuh), output positions
// come from a block scan plus the single-pass ordered tile prefix in ak_scan.cuh, so the text is read from HBM
// once and every output is written once.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <exception>
#include <new>
#include <string>
#include <vector>

#include "../../include/akshar_b200.h"
#include "ak_models.h"
#include "ak_scan.cuh"
#include "ak_subword.cuh"
#include "ak_fast.cuh"
#include "ak_norm3.cuh"
#include "ak_seg3.cuh"
#include "ak_bpe3.cuh"
#include "ak_tok.cuh"
#include "ak_tok_host.h"
#include "ak_decode_host.h"
#include "unicode_tables.inc"


#include "ak_common.cuh"
#include "ak_norm_kernels.cuh"
#include "ak_seg_kernels.cuh"
#include "ak_sub_kernels.cuh"
#include "ak_tok_kernels.cuh"
#include "ak_wtok_kernels.cuh"
#include "ak_decode_kernels.cuh"
#include "ak_feat_kernels.cuh"
#include "ak_lines_kernels.cuh"
#include "ak_win_kernels.cuh"
#include "ak_pair_kernels.cuh"
#include "ak_pack_kernels.cuh"

// ================================================================================================
// host side: context, model upload, C ABI
// ================================================================================================
struct AkcTable {
    AkWordCache work{};
    unsigned long long* image = nullptr;
    size_t bytes = 0;
    bool reset = false;            // restore the image at the next call whatever the fill
};

struct akshar_ctx {
    int device = 0;
    int sm_count = 148;
    AkTables T{};
    std::vector<void*> allocs;
    std::string err;
    int64_t launches = 0;
    bool has_bpe = false, has_uni = false;
    AkBpeHost bpe_h;
    AkBpeDev bpe_d{};
    AkUniHost uni_h;
    AkUniDev uni_d{};
    std::vector<void*> bpe_allocs, uni_allocs;
    // event-stream encoders (ak_tok.cuh): one word cache per model, image built at load
    AkcTable tok_cache[2];
    AkDecTable dec[2][2] = {};     // [kind][form]: piece tables of the on-device decode / detokenize (ak_decode.cuh)
    bool uni_fast = false;         // the Unigram model has the shape the word-wise path needs
    int occ_words[2] = {0, 0}, occ_resolve[2] = {0, 0}, occ_check = 0, occ_emit = 0;
    // optional CUDA-event timing of the dominant kernel of each stage (bench.py's roofline line)
    bool timing = false;
    bool wc_hold = false;          // akshar_word_cache_hold(1): never restore the image, however full the cache
    cudaEvent_t tev[AKSHAR_TIMER_COUNT][2] = {};
    bool tev_valid[AKSHAR_TIMER_COUNT] = {};
    int occ_norm = 0, occ_seg = 0, occ_uni = 0, occ_sig = 0, occ_nf_write = 0, occ_nf3 = 0;
};

// the entry points run on the context's device and leave the caller's current device as they found it
struct AkDeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit AkDeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
    }
    ~AkDeviceGuard() {
        if (switched) cudaSetDevice(prev);
    }
};

#define AK_CUDA(ctx, call)                                                                         \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                       \
            return AKSHAR_E_CUDA;                                                                  \
        }                                                                                          \
    } while (0)

template <class V>
static int ak_upload(akshar_ctx* ctx, std::vector<void*>& owner, const V* src, size_t n, const V** dst) {
    void* d = nullptr;
    size_t bytes = (n ? n : 1) * sizeof(V);
    AK_CUDA(ctx, cudaMalloc(&d, bytes));
    owner.push_back(d);
    if (n) AK_CUDA(ctx, cudaMemcpy(d, src, n * sizeof(V), cudaMemcpyHostToDevice));
    *dst = (const V*)d;
    return 0;
}

extern "C" {

int akshar_version(void) { return 100; }

const char* akshar_status_str(int code) {
    switch (code) {
        case AKSHAR_OK: return "ok";
        case AKSHAR_E_ARG: return "bad argument";
        case AKSHAR_E_CUDA: return "CUDA error";
        case AKSHAR_E_MODEL: return "model could not be parsed or uses an unsupported configuration";
        case AKSHAR_E_NOMODEL: return "no model loaded for this encoder";
        case AKSHAR_E_WORKSPACE: return "workspace too small";
        default: return "unknown";
    }
}

int akshar_ctx_create(int device, akshar_ctx** out) {
    if (!out) return AKSHAR_E_ARG;
    *out = nullptr;
    akshar_ctx* ctx = new (std::nothrow) akshar_ctx();
    if (!ctx) return AKSHAR_E_ARG;
    ctx->device = device;
    *out = ctx;      // returned even on failure so that akshar_last_error can be read; caller destroys it
    AkDeviceGuard device_guard(device);
    AK_CUDA(ctx, cudaSetDevice(device));
    cudaDeviceProp prop;
    AK_CUDA(ctx, cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        ctx->err = "akshar_b200 is built for sm_100a (B200); device is sm_" + std::to_string(prop.major * 10 + prop.minor);
        return AKSHAR_E_CUDA;
    }
    ctx->sm_count = prop.multiProcessorCount;
    int rc;
#define UP(field, arr, n, type) \
    if ((rc = ak_upload<type>(ctx, ctx->allocs, (const type*)(arr), (size_t)(n), (const type**)&ctx->T.field))) return rc;
    UP(page_index, ak_tbl_page_index, AK_N_PAGES, uint16_t)
    UP(leaves, ak_tbl_leaves, AK_N_LEAF_PAGES * 256, uint32_t)
    UP(decomp_keys, ak_tbl_decomp_keys, AK_N_DECOMP, uint32_t)
    UP(decomp_off, ak_tbl_decomp_off, AK_N_DECOMP + 1, uint16_t)
    UP(decomp_data, ak_tbl_decomp_data, AK_N_DECOMP_DATA, uint32_t)
    UP(pair_keys, ak_tbl_pair_keys, AK_N_PAIRS, unsigned long long)
    UP(pair_vals, ak_tbl_pair_vals, AK_N_PAIRS, uint32_t)
    UP(ll_keys, ak_tbl_latin_lower_keys, AK_N_LATIN_LOWER, uint32_t)
    UP(ll_vals, ak_tbl_latin_lower_vals, AK_N_LATIN_LOWER, uint32_t)
    UP(fl_keys, ak_tbl_full_lower_keys, AK_N_FULL_LOWER, uint32_t)
    UP(fl_vals, ak_tbl_full_lower_vals, AK_N_FULL_LOWER, uint32_t)
    UP(kmap_keys, ak_tbl_kmap_keys, AK_N_KMAP, uint32_t)
    UP(kmap_off, ak_tbl_kmap_off, AK_N_KMAP + 1, uint16_t)
    UP(kmap_data, ak_tbl_kmap_data, AK_N_KMAP_DATA, uint32_t)
    UP(hf_unknown, ak_tbl_hf_unknown, AK_N_HF_UNKNOWN, uint32_t)
#undef UP
    ctx->T.n_decomp = AK_N_DECOMP;
    ctx->T.n_pairs = AK_N_PAIRS;
    ctx->T.n_ll = AK_N_LATIN_LOWER;
    ctx->T.n_fl = AK_N_FULL_LOWER;
    ctx->T.n_kmap = AK_N_KMAP;
    ctx->T.n_hf_unknown = AK_N_HF_UNKNOWN;
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_norm, ak_normalize_kernel, AK_BLOCK, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_nf_write, ak_nf_write_kernel, AK_BLOCK, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_nf3, ak_nf3_classify_kernel, AKN3_THREADS, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_seg, ak_segment_kernel, AK_BLOCK, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_uni, ak_unigram_kernel, AK_ROWS_BLOCK, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_sig, ak_signature_kernel, AK_ROWS_BLOCK, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_words[0], ak_words_kernel<0>, AKW_THREADS, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_words[1], ak_words_kernel<1>, AKW_THREADS, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_resolve[0], ak_resolve_kernel<0>, AKR_THREADS, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_resolve[1], ak_resolve_kernel<1>, AKR_THREADS, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_check, ak_unicheck_kernel, AKL_THREADS, 0));
    AK_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ_emit, ak_emit_kernel<int32_t>, AKL_THREADS, 0));
    return AKSHAR_OK;
}

static void ak_free_list(std::vector<void*>& v) {
    for (void* p : v) cudaFree(p);
    v.clear();
}

void akshar_ctx_destroy(akshar_ctx* ctx) {
    if (!ctx) return;
    AkDeviceGuard device_guard(ctx->device);
    ak_free_list(ctx->allocs);
    ak_free_list(ctx->bpe_allocs);
    ak_free_list(ctx->uni_allocs);
    for (int i = 0; i < AKSHAR_TIMER_COUNT; ++i)
        for (int k = 0; k < 2; ++k)
            if (ctx->tev[i][k]) cudaEventDestroy(ctx->tev[i][k]);
    delete ctx;
}

const char* akshar_last_error(akshar_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int akshar_word_cache_hold(akshar_ctx* ctx, int hold) {
    if (!ctx) return AKSHAR_E_ARG;
    if (hold < 0) {
        ctx->tok_cache[0].reset = ctx->tok_cache[1].reset = true;
        return AKSHAR_OK;
    }
    ctx->wc_hold = hold != 0;
    return AKSHAR_OK;
}

int akshar_timing_enable(akshar_ctx* ctx, int enable) {
    AkDeviceGuard device_guard(ctx ? ctx->device : 0);
    if (!ctx) return AKSHAR_E_ARG;
    AK_CUDA(ctx, cudaSetDevice(ctx->device));
    if (enable)
        for (int i = 0; i < AKSHAR_TIMER_COUNT; ++i)
            for (int k = 0; k < 2; ++k)
                if (!ctx->tev[i][k]) AK_CUDA(ctx, cudaEventCreate(&ctx->tev[i][k]));
    ctx->timing = enable != 0;
    for (int i = 0; i < AKSHAR_TIMER_COUNT; ++i) ctx->tev_valid[i] = false;
    return AKSHAR_OK;
}

int akshar_timing_read(akshar_ctx* ctx, int timer, float* ms) {
    if (!ctx || !ms || timer < 0 || timer >= AKSHAR_TIMER_COUNT) return AKSHAR_E_ARG;
    if (!ctx->tev_valid[timer]) return AKSHAR_E_ARG;
    AK_CUDA(ctx, cudaEventSynchronize(ctx->tev[timer][1]));
    AK_CUDA(ctx, cudaEventElapsedTime(ms, ctx->tev[timer][0], ctx->tev[timer][1]));
    return AKSHAR_OK;
}

int64_t akshar_launch_count(akshar_ctx* ctx) { return ctx ? ctx->launches : 0; }

// workspace layout (all regions 256-byte aligned):
//   [0, 256)            control block: tickets[8] (int), changed flag, pool cursor
//   state regions       4 x n_tiles x 8 bytes (two counters x two passes)
//   scratch             max(unigram back-pointers 4 (n_bytes + 2 n_rows + 2), signature code points 4 n_bytes,
//                           BPE: NFC'd text n_bytes + n_bytes / 8 + 1024, its row offsets 8 (n_rows + 1), long-word pool)
static inline size_t ak_align(size_t x) { return (x + 255) & ~(size_t)255; }
static inline int64_t ak_tiles_of(int64_t n_bytes, int64_t n_rows) {
    int64_t a = (n_bytes + n_bytes / 8 + 1024 + 32 + AKF_TILE - 1) / AKF_TILE;     // fast-kernel tiles; covers the NFC'd copy too
    int64_t b = (n_rows + AK_ROWS_BLOCK - 1) / AK_ROWS_BLOCK;
    return (a > b ? a : b) + 1;
}
struct AkTokWs {
    size_t wrow, count, wt_ids, wt_base, wt_seg, wt_segx, scan_state, row_flag, row_ev, row_fix, pool, longpool, slots, total;
    size_t pool_ints, longpool_ints;
    int64_t n_wt;
};
#define AKT_CAP_MIN 256            // event slots per 960 text bytes with the minimum workspace (0.27 events per byte)
#define AKT_CAP_MAX 2048           // a row start and a word start at every byte: 1920
#define AKT_SLOT_BYTES 20          // event + resolved record + aux word
static AkTokWs ak_tok_ws(int64_t n_bytes, int64_t n_rows) {
    AkTokWs W;
    W.n_wt = n_bytes / AKT_WARP_BYTES + 3;
    size_t at = 0;
    W.wrow = at;       at += ak_align(((size_t)W.n_wt * 2 + 4) * 8);
    W.count = at;      at += ak_align((size_t)W.n_wt * 4);
    W.wt_ids = at;     at += ak_align((size_t)W.n_wt * 4);
    W.wt_base = at;    at += ak_align((size_t)W.n_wt * 8);
    W.wt_seg = at;     at += ak_align((size_t)W.n_wt * 8);
    W.wt_segx = at;    at += ak_align((size_t)W.n_wt * 4);
    W.scan_state = at; at += 2 * ak_align(((size_t)W.n_wt / AKS_TILE + 2) * 8);
    W.row_flag = at;   at += ak_align((size_t)n_rows + 1);
    W.row_ev = at;     at += ak_align(((size_t)n_rows + 2) * 4);
    W.row_fix = at;    at += ak_align(((size_t)n_rows + 1) * 8);
    W.pool_ints = (size_t)n_bytes / 4 + 65536;
    W.pool = at;       at += ak_align(W.pool_ints * 4);
    W.longpool_ints = (size_t)n_bytes / 8 + 65536;
    W.longpool = at;   at += ak_align(W.longpool_ints * 4);
    W.slots = at;      // events, resolved records, aux words: sized at run time from the real workspace
    at += (size_t)W.n_wt * AKT_CAP_MIN * (AKT_SLOT_BYTES + 1) + 8192;
    W.total = at;
    return W;
}

struct AkWsLayout {
    size_t control, state, tile_row, scratch, total;
};
// [0, 256) control block, then the zeroed tile-state area (look-back states of the walker kernels, scan states), the
// tile -> row table of the normalize kernels, and a scratch region shared by whatever stage runs: its size is the largest
// any entry point needs for this text
static AkWsLayout ak_ws_layout(int64_t n_bytes, int64_t n_rows) {
    AkWsLayout L;
    size_t tiles = (size_t)ak_tiles_of(n_bytes, n_rows);
    L.control = 0;
    L.state = 256;
    L.tile_row = L.state + ak_align(4 * tiles * 8);
    size_t at = L.tile_row + ak_align(8 * (tiles * AKF_WARPS + 2));
    L.scratch = at;
    // Unigram row kernel / signatures: one 4-byte slot per code point (+ 2 per row)
    size_t m = 4 * (size_t)(n_bytes + 2 * n_rows + 2);
    // fast normalize: per-lane info words, tile totals / bases, slow work list
    const size_t nf = ak_align(tiles * AK_BLOCK * 4) + ak_align(tiles * AKF_WARPS * 4) + ak_align((tiles * AKF_WARPS + 1) * 8) +
                      ak_align((tiles * AK_BLOCK / 16 + 1024) * sizeof(AkSlowEntry));
    if (nf > m) m = nf;
    // segment / word tokenizers: warp-tile row table, two counts and two bases per 960-byte warp tile
    const size_t n_wt = (size_t)n_bytes / AKN3_WARP_BYTES + 3;
    const size_t sg = ak_align((2 * n_wt + 3) * 8) + 2 * ak_align(n_wt * 4) + 2 * ak_align(n_wt * 8);
    if (sg > m) m = sg;
    const size_t tok = ak_tok_ws(n_bytes, n_rows).total;
    if (tok > m) m = tok;
    L.total = at + ak_align(m);
    return L;
}

size_t akshar_workspace_bytes(int64_t n_bytes, int64_t n_rows) {
    if (n_bytes < 0 || n_rows < 0) return 0;
    return ak_ws_layout(n_bytes, n_rows).total;
}

struct AkCall {
    akshar_ctx* ctx;
    AkBatch B;
    AkWsLayout L;
    char* ws;
    size_t ws_bytes;       // what the caller really passed: the temporary streams use everything beyond the fixed part
    cudaStream_t stream;
};

// validates the common arguments, clears the control block + result, fills AkBatch (tiles for `mode`)
static int ak_begin(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows, int64_t text_begin,
                    int64_t text_end, int mode, int rows_block, int64_t* d_result, void* d_workspace, size_t workspace_bytes,
                    void* stream, AkCall& C) {
    if (!ctx) return AKSHAR_E_ARG;
    if (!d_row_offsets || !d_result || n_rows < 0 || text_end < text_begin || (!d_text && text_end > text_begin) ||
        (mode != AKSHAR_MODE_TILES && mode != AKSHAR_MODE_ROWS)) {
        ctx->err = "bad argument";
        return AKSHAR_E_ARG;
    }
    const int64_t n_bytes = text_end - text_begin;
    // positions inside a call are 32-bit (event records, tile-relative offsets) and a row index shares a 32-bit word with
    // three kind bits: larger inputs are fed as several calls (row ranges keep their absolute offsets: text_begin / text_end)
    if (n_bytes >= AKSHAR_MAX_CALL_BYTES || n_rows >= AKSHAR_MAX_CALL_ROWS) {
        ctx->err = "batch too large for one call: at most 4 GiB - 64 KiB of text and 2^29 - 1 rows; split it by row ranges";
        return AKSHAR_E_ARG;
    }
    C.ctx = ctx;
    C.L = ak_ws_layout(n_bytes, n_rows);
    if (!d_workspace || workspace_bytes < C.L.total) {
        ctx->err = "workspace too small: need " + std::to_string(C.L.total) + " bytes";
        return AKSHAR_E_WORKSPACE;
    }
    C.ws = (char*)d_workspace;
    C.ws_bytes = workspace_bytes;
    C.stream = (cudaStream_t)stream;
    AK_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t tiles = (size_t)ak_tiles_of(n_bytes, n_rows);
    AK_CUDA(ctx, cudaMemsetAsync(C.ws, 0, 256 + ak_align(4 * tiles * 8), C.stream));
    AK_CUDA(ctx, cudaMemsetAsync(d_result, 0, 4 * sizeof(int64_t), C.stream));
    AkBatch& B = C.B;
    B.text = d_text;
    B.off = d_row_offsets;
    B.n_rows = n_rows;
    B.text_begin = text_begin;
    B.text_end = text_end;
    B.mode = mode;
    if (rows_block > 0) B.n_tiles = (int)((n_rows + rows_block - 1) / rows_block);
    else if (mode == AKSHAR_MODE_TILES) B.n_tiles = (int)((n_bytes + 1 + AK_TILE - 1) / AK_TILE);
    else B.n_tiles = (int)((n_rows + AK_BLOCK - 1) / AK_BLOCK);
    B.ticket = (int*)C.ws;
    B.state0 = (unsigned long long*)(C.ws + C.L.state);
    B.state1 = B.state0 + tiles;
    B.result = d_result;
    B.totals = d_result;
    B.run_if = nullptr;
    B.dyn_end = nullptr;
    return AKSHAR_OK;
}

// brackets one kernel launch with events when timing is enabled
struct AkTimed {
    akshar_ctx* ctx;
    int slot;
    cudaStream_t s;
    AkTimed(akshar_ctx* c, int sl, cudaStream_t st) : ctx(c), slot(sl), s(st) {
        if (ctx->timing && ctx->tev[slot][0]) cudaEventRecord(ctx->tev[slot][0], s);
    }
    ~AkTimed() {
        if (ctx->timing && ctx->tev[slot][1]) { cudaEventRecord(ctx->tev[slot][1], s); ctx->tev_valid[slot] = true; }
    }
};

static int ak_grid(akshar_ctx* ctx, int occ, int n_tiles) {
    int g = ctx->sm_count * (occ > 0 ? occ : 1);
    return n_tiles < g ? (n_tiles > 0 ? n_tiles : 1) : g;
}

static int ak_after_launch(akshar_ctx* ctx, const char* what) {
    cudaError_t e = cudaGetLastError();
    // AKSHAR_DEBUG_SYNC=1: wait for every kernel and say which one faulted (debugging aid; never set in production)
    static const bool debug_sync = getenv("AKSHAR_DEBUG_SYNC") != nullptr;
    if (e == cudaSuccess && debug_sync) {
        e = cudaDeviceSynchronize();
        if (e != cudaSuccess) fprintf(stderr, "akshar_b200: kernel '%s' failed: %s\n", what, cudaGetErrorString(e));
    }
    if (e != cudaSuccess) {
        ctx->err = std::string(what) + " launch: " + cudaGetErrorString(e);
        return AKSHAR_E_CUDA;
    }
    ctx->launches++;
    return AKSHAR_OK;
}

// a batch with no rows: every ragged output is just splits[0] = 0
static int ak_empty_rows(akshar_ctx* ctx, int64_t* a, int64_t* b, cudaStream_t s) {
    if (a) AK_CUDA(ctx, cudaMemsetAsync(a, 0, sizeof(int64_t), s));
    if (b) AK_CUDA(ctx, cudaMemsetAsync(b, 0, sizeof(int64_t), s));
    return AKSHAR_OK;
}

#include "ak_abi_text.inc"

}  // extern "C"

#include "ak_abi_aux.inc"
#include "ak_abi_models.inc"
#include "ak_abi_encode.inc"
