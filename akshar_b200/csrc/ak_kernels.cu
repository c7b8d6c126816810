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

#include <algorithm>
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
#include "ak_mlm_kernels.cuh"

// ================================================================================================
// host side: context, model upload, C ABI
// ================================================================================================
struct AkcTable {
    AkWordCache work{};
    unsigned long long* image = nullptr;
    size_t bytes = 0;
    int64_t image_entries = 0;     // entries of the image built at load
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
    const uint32_t* mlm_special[2] = {};  // [kind]: one bit per id of the model's special ids (akshar_mlm_mask)
    int64_t mlm_bits[2] = {0, 0};
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

// sets the text akshar_last_error returns and passes the status code on
static int ak_fail(akshar_ctx* ctx, int code, std::string msg) {
    ctx->err = std::move(msg);
    return code;
}

static int ak_ws_short(akshar_ctx* ctx, size_t need) {
    return ak_fail(ctx, AKSHAR_E_WORKSPACE, "workspace too small: need " + std::to_string(need) + " bytes");
}

// calls f with a value of the caller's id type: uint16_t when ids_u16, int32_t otherwise
template <class F>
static int ak_with_ids(int ids_u16, F f) {
    return ids_u16 ? f(uint16_t()) : f(int32_t());
}

static inline size_t ak_align(size_t x) { return (x + 255) & ~(size_t)255; }
// the tile states of one ak_scan_counts_kernel over at most n entries
static inline size_t ak_scan_state_bytes(size_t n) { return ak_align((n / AKS_TILE + 2) * 8); }

// Bump allocator of one workspace layout: every region starts 256-byte aligned.  With a null base it only adds up the
// sizes, so one function both sizes a workspace (akshar_*_workspace_bytes, ak_ws_layout) and carves it (the launcher).
struct AkCarve {
    char* base;
    size_t at;
    template <class T>
    void take(T*& p, size_t bytes) {
        p = base ? (T*)(base + at) : nullptr;
        at += ak_align(bytes);
    }
};

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
    if (prop.major < 10)
        return ak_fail(ctx, AKSHAR_E_CUDA, "akshar_b200 is built for sm_100a (B200); device is sm_" + std::to_string(prop.major * 10 + prop.minor));
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

int akshar_word_cache_stats(akshar_ctx* ctx, int kind, int64_t* out, void* stream) {
    if (!ctx || !out || (kind != 0 && kind != 1)) return AKSHAR_E_ARG;
    // the Unigram encoder has a word cache only with the word-wise model shape
    if (kind == 0 ? !ctx->has_bpe : !(ctx->has_uni && ctx->uni_fast)) return AKSHAR_E_NOMODEL;
    AkDeviceGuard device_guard(ctx->device);
    const AkcTable& t = ctx->tok_cache[kind];
    unsigned long long learned = 0;
    AK_CUDA(ctx, cudaMemcpyAsync(&learned, t.work.inserted, sizeof(learned), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    AK_CUDA(ctx, cudaStreamSynchronize((cudaStream_t)stream));
    out[0] = (int64_t)1 << t.work.bits;
    out[1] = t.image_entries;
    out[2] = (int64_t)learned;
    out[3] = ctx->wc_hold ? 1 : 0;
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

// The first 256 bytes of every workspace, zeroed by each call before its first kernel.  A ticket hands out tile numbers
// in the order the CTAs ask, so no two stages of one call may share one: the second would start at the first one's last
// tile and skip the tiles before it.  The fused calls run the normalize stage (ticket or scan_b, n_slow) and then the
// segment mask kernel (no control word) or an encoder (uni_rows, or scan_a, seg_scan and the event-stream words).
struct AkControl {
    int ticket;                      // tile ticket (AkBatch::ticket) of the walker kernels: generic normalize, generic
                                     // segment, signatures; the scan ticket of decode, merge, lines, windows, pairs, pack
    int uni_rows;                    // Unigram row kernel
    int seg_scan;                    // event-stream Unigram: segmented scan
    int scan_a;                      // scans: segment offsets' clusters, word tokenizer, event-stream encoders' ids
    int scan_b;                      // scans: segment offsets' runs, fast normalize's output bytes
    unsigned int n_slow;             // fast normalize: entries of the slow-lane work list
    unsigned int any_flag;           // event-stream encoders: some row goes to the row-fix kernel
    long long n_wt;                  // event-stream encoders: warp tiles the words kernel found (the scans' count)
    unsigned long long longpool_used;  // event-stream encoders: long-word pool cursor
    unsigned long long pool_used;    // event-stream encoders: id / Viterbi scratch pool cursor
    unsigned long long pair_windows; // pair windows count: the windows of all pairs,
    unsigned int pair_done;          // the blocks that have added theirs,
    long long pair_n_scan;           // and the entries the scan takes (0 when the total does not fit its 32-bit tile sums)
    int64_t pack_pieces;             // pack count: the scan's total
};
static_assert(sizeof(AkControl) <= 256, "the control block is the first 256 bytes of a workspace");

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
    W.scan_state = at; at += 2 * ak_scan_state_bytes((size_t)W.n_wt);
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

// Scratch layouts of the text stages.  Each returns its size and, given a base, carves it; the launcher passes the tiles
// it really has, ak_ws_layout the most the text can have.
// fast normalize: per-lane info words, warp-tile totals and bases, the slow-lane work list
static size_t ak_nf_ws(size_t n_tiles, char* base, AkNfWork& W) {
    AkCarve c{base, 0};
    c.take(W.info, n_tiles * AK_BLOCK * 4);
    c.take(W.tile_total, n_tiles * AKF_WARPS * 4);
    c.take(W.tile_base, (n_tiles * AKF_WARPS + 1) * 8);
    const size_t slow_cap = n_tiles * AK_BLOCK / 16 + 1024;
    W.slow_cap = (unsigned int)slow_cap;
    c.take(W.slow, slow_cap * sizeof(AkSlowEntry));
    return c.at;
}
// segment offsets: warp-tile row table, cluster and run counts and their bases per warp tile
struct AkSegWs {
    int64_t* wrow;
    int32_t *c_count, *r_count;
    int64_t *c_base, *r_base;
};
static size_t ak_seg_ws(size_t n_wt, char* base, AkSegWs& W) {
    AkCarve c{base, 0};
    c.take(W.wrow, (n_wt * 2 + 3) * 8);
    c.take(W.c_count, n_wt * 4);
    c.take(W.r_count, n_wt * 4);
    c.take(W.c_base, n_wt * 8);
    c.take(W.r_base, n_wt * 8);
    return c.at;
}
// segment masks: the warp-tile row table
static size_t ak_seg_mask_ws(size_t n_wt, char* base, int64_t*& wrow) {
    AkCarve c{base, 0};
    c.take(wrow, (n_wt * 2 + 3) * 8);
    return c.at;
}
// word tokenizers: warp-tile row table, word counts and their bases per warp tile
struct AkWtWs {
    int64_t* wrow;
    int32_t* count;
    int64_t* base;
};
static size_t ak_wt_ws(size_t n_wt, char* base, AkWtWs& W) {
    AkCarve c{base, 0};
    c.take(W.wrow, (n_wt * 2 + 3) * 8);
    c.take(W.count, n_wt * 4);
    c.take(W.base, n_wt * 8);
    return c.at;
}

struct AkWsLayout {
    size_t state, tile_row, scratch, total;
};
// [0, 256) control block, then the zeroed tile-state area (look-back states of the walker kernels, scan states), the
// tile -> row table of the normalize kernels, and a scratch region shared by whatever stage runs: its size is the largest
// any entry point needs for this text
static AkWsLayout ak_ws_layout(int64_t n_bytes, int64_t n_rows) {
    AkWsLayout L;
    size_t tiles = (size_t)ak_tiles_of(n_bytes, n_rows);
    L.state = 256;
    L.tile_row = L.state + ak_align(4 * tiles * 8);
    L.scratch = L.tile_row + ak_align(8 * (tiles * AKF_WARPS + 2));
    // Unigram row kernel / signatures: one 4-byte slot per code point (+ 2 per row)
    const size_t rows = 4 * (size_t)(n_bytes + 2 * n_rows + 2);
    const size_t n_wt = (size_t)n_bytes / AKN3_WARP_BYTES + 3, n_wt_words = (size_t)n_bytes / AKT_WARP_BYTES + 3;
    AkNfWork nf;
    AkSegWs sg;
    int64_t* wrow;
    AkWtWs wt;
    const size_t m = std::max({rows, ak_nf_ws(tiles, nullptr, nf), ak_seg_ws(n_wt, nullptr, sg), ak_seg_mask_ws(n_wt, nullptr, wrow),
                               ak_wt_ws(n_wt_words, nullptr, wt), ak_tok_ws(n_bytes, n_rows).total});
    L.total = L.scratch + ak_align(m);
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
    AkControl* K;          // the workspace's control block
    size_t ws_bytes;       // what the caller really passed: the temporary streams use everything beyond the fixed part
    cudaStream_t stream;
};

// validates the common arguments, clears the control block, the tile states and the result, fills AkBatch (tiles for
// `mode`).  The workspace is laid out for the larger of the text and layout_bytes: a fused call passes the capacity of
// the normalized text its second stage reads.
static int ak_begin(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows, int64_t text_begin,
                    int64_t text_end, int64_t layout_bytes, int mode, int rows_block, int64_t* d_result, void* d_workspace,
                    size_t workspace_bytes, void* stream, AkCall& C) {
    if (!ctx) return AKSHAR_E_ARG;
    if (!d_row_offsets || !d_result || n_rows < 0 || text_end < text_begin || (!d_text && text_end > text_begin) ||
        (mode != AKSHAR_MODE_TILES && mode != AKSHAR_MODE_ROWS))
        return ak_fail(ctx, AKSHAR_E_ARG, "bad argument");
    const int64_t n_bytes = text_end - text_begin;
    // positions inside a call are 32-bit (event records, tile-relative offsets) and a row index shares a 32-bit word with
    // three kind bits: larger inputs are fed as several calls (row ranges keep their absolute offsets: text_begin / text_end)
    if (n_bytes >= AKSHAR_MAX_CALL_BYTES || n_rows >= AKSHAR_MAX_CALL_ROWS)
        return ak_fail(ctx, AKSHAR_E_ARG,
                       "batch too large for one call: at most 4 GiB - 64 KiB of text and 2^29 - 1 rows; split it by row ranges");
    const int64_t lay = layout_bytes > n_bytes ? layout_bytes : n_bytes;
    C.ctx = ctx;
    C.L = ak_ws_layout(lay, n_rows);
    if (!d_workspace || workspace_bytes < C.L.total) return ak_ws_short(ctx, C.L.total);
    C.ws = (char*)d_workspace;
    C.K = (AkControl*)C.ws;
    C.ws_bytes = workspace_bytes;
    C.stream = (cudaStream_t)stream;
    AK_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t tiles = (size_t)ak_tiles_of(lay, n_rows);
    AK_CUDA(ctx, cudaMemsetAsync(C.ws, 0, C.L.tile_row, C.stream));
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
    B.ticket = &C.K->ticket;
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
    if (e != cudaSuccess) return ak_fail(ctx, AKSHAR_E_CUDA, std::string(what) + " launch: " + cudaGetErrorString(e));
    ctx->launches++;
    return AKSHAR_OK;
}

// exclusive prefix sums of the n int32 counts v into base, their sum into *total (ak_scan.cuh), status bits into result[2].
// With n_dyn the count is only known on the device and n bounds it.  Each scan of a call has its own ticket and tile states.
static int ak_scan_counts(akshar_ctx* ctx, cudaStream_t s, const char* what, const int32_t* v, long long n, const long long* n_dyn,
                          int64_t* base, int64_t* total, int* ticket, unsigned long long* state, int64_t* result) {
    ak_scan_counts_kernel<<<ak_grid(ctx, 4, (int)(n / AKS_TILE + 1)), AKS_THREADS, 0, s>>>(v, n_dyn ? 0 : n, n_dyn, 1, base, total, ticket,
                                                                                          state, (unsigned int*)&result[2]);
    return ak_after_launch(ctx, what);
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
