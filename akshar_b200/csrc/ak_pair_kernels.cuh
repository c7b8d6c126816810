// Kernels of the model-ready sentence-pair windows (two ragged id sets -> input_ids / attention_mask [N, L], HF
// tokenizers' pair truncation with stride + the pair template + padding; include/akshar_b200.h,
// akshar_pair_windows_count / akshar_pair_windows_write).  The per-pair arithmetic is akpair_plan (ak_win.cuh).
//   ak_pair_count_kernel   one thread per pair: the template check of both rows, its window count wa * wb, the longest
//                          window (always window (0, 0)), the lowest refused pair
//   (ak_scan_counts_kernel) window splits of the pairs, N
//   ak_pair_write_kernel   one warp per window: its pair by the 32-way search of the single windows (akwin_owner), its
//                          (i, j), then pre + A_i + mid + B_j + post and the pads as coalesced int64 stores
#pragma once
#include "ak_win_kernels.cuh"

#define AKPAIR_SLOT 4                  // ids per slot of the pair template

template <class IdT>
struct AkPairArgs {
    const IdT* ids_a;
    const int64_t* splits_a;           // [n_pairs + 1] positions in ids_a
    const IdT* ids_b;
    const int64_t* splits_b;           // [n_pairs + 1] positions in ids_b
    int64_t n_pairs;
    int32_t bos, eos;                  // ids of the single template around every row, -1: none
    int32_t tmpl[3 * AKPAIR_SLOT];     // pair template: pre, mid, post slots of AKPAIR_SLOT ids
    int32_t n_pre, n_mid, n_post;
    int64_t m;                         // content budget: max_length - (n_pre + n_mid + n_post)
    int64_t stride;
    int strategy;                      // AKPAIR_NONE, AKPAIR_LONGEST_FIRST, AKPAIR_ONLY_FIRST, AKPAIR_ONLY_SECOND
    bool overflow, left, pad_left;
};

// content [lo, lo + c) of a row framed by the single template; false when it is not framed
template <class IdT>
__device__ __forceinline__ bool akpair_content(const AkPairArgs<IdT>& A, const IdT* ids, const int64_t* splits, int64_t r, int64_t& lo,
                                               int64_t& c) {
    const int head = A.bos >= 0, s = head + (A.eos >= 0);
    const int64_t b = splits[r], e = splits[r + 1], n = e - b;
    lo = b + head;
    c = n > s ? n - s : 0;
    return !(n < s || (A.bos >= 0 && (int32_t)ids[b] != A.bos) || (A.eos >= 0 && (int32_t)ids[e - 1] != A.eos));
}

// the windows of the whole call, which the count kernel adds up in 64 bits: a single pair is refused above 2^31 - 1
// windows, but several pairs under that bound can still sum past what the scan's 32-bit tile sums hold
struct AkPairTotal {
    unsigned long long* windows;       // zeroed
    unsigned int* done;                // zeroed: blocks that have added their windows
    long long* n_scan;                 // written by the last block: n_pairs + 1 entries to scan, or 0 when the call is refused
};

// count[p] = windows of pair p (count[n_pairs] = 0); result[1] = longest window; result[2] |= AKSHAR_ST_TEMPLATE /
// AKSHAR_ST_PAIR_TRUNC; result[3] = min over refused pairs of pair * 8 + reason (all ones: none), and
// n_pairs * 8 + AKPAIR_CALL_TOO_MANY when the pairs give more than 2^31 - 1 windows in all
template <class IdT>
__global__ void __launch_bounds__(AKWIN_THREADS) ak_pair_count_kernel(const AkPairArgs<IdT> A, int32_t* count, int64_t* result,
                                                                      const AkPairTotal T) {
    const int64_t P = A.n_pre + A.n_mid + A.n_post;
    unsigned long long longest = 0, refused = ~0ull, windows = 0;
    uint32_t st = 0;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= A.n_pairs; r += (int64_t)gridDim.x * blockDim.x) {
        if (r == A.n_pairs) {
            count[r] = 0;
            continue;
        }
        int64_t la, ca, lb, cb;
        if (!akpair_content(A, A.ids_a, A.splits_a, r, la, ca) || !akpair_content(A, A.ids_b, A.splits_b, r, lb, cb)) st |= AKSHAR_ST_TEMPLATE;
        const AkPairPlan p = akpair_plan(ca, cb, A.m, A.stride, A.strategy, A.overflow);
        if (p.reason) {
            st |= AKSHAR_ST_PAIR_TRUNC;
            const unsigned long long code = (unsigned long long)r * 8 + (unsigned)p.reason;
            refused = code < refused ? code : refused;
            count[r] = 1;
            ++windows;
            continue;
        }
        count[r] = (int32_t)(p.wa * p.wb);
        windows += (unsigned long long)(p.wa * p.wb);
        const unsigned long long len = (unsigned long long)(P + p.na + p.nb);
        longest = len > longest ? len : longest;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, longest, d);
        longest = o > longest ? o : longest;
        const unsigned long long q = __shfl_xor_sync(0xFFFFFFFFu, refused, d);
        refused = q < refused ? q : refused;
        st |= __shfl_xor_sync(0xFFFFFFFFu, st, d);
        windows += __shfl_xor_sync(0xFFFFFFFFu, windows, d);
    }
    if ((threadIdx.x & 31) == 0) {
        if (longest) atomicMax((unsigned long long*)&result[1], longest);
        if (st) atomicOr((unsigned int*)&result[2], st);
        if (refused != ~0ull) atomicMin((unsigned long long*)&result[3], refused);
        if (windows) atomicAdd(T.windows, windows);
    }
    // the last block to finish sees every block's windows (threadfence reduction)
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(T.done, 1u) == gridDim.x - 1) {
        __threadfence();
        if (atomicAdd(T.windows, 0ull) > (unsigned long long)INT32_MAX) {
            atomicOr((unsigned int*)&result[2], (unsigned int)AKSHAR_ST_PAIR_TRUNC);
            atomicMin((unsigned long long*)&result[3], (unsigned long long)A.n_pairs * 8 + AKPAIR_CALL_TOO_MANY);
            *T.n_scan = 0;
        } else {
            *T.n_scan = A.n_pairs + 1;
        }
    }
}

// one warp per window; as in ak_win_write_kernel the loads of AKWIN_UNROLL positions are issued before their stores.
// A position is a content id of A or B (one predicated load from either side), a template id (from shared memory) or a pad
template <class IdT>
__global__ void __launch_bounds__(AKWIN_THREADS) ak_pair_write_kernel(const AkPairArgs<IdT> A, const int64_t* __restrict__ wsplits,
                                                                      int64_t n_windows, int64_t width, int64_t pad_id,
                                                                      int64_t* __restrict__ out_ids, int64_t* __restrict__ out_mask,
                                                                      int64_t* __restrict__ sample) {
    __shared__ int32_t s_tmpl[16];                            // the 3 slots, then 4 unused entries
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < 3 * AKPAIR_SLOT; ++i) s_tmpl[i] = A.tmpl[i];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (AKWIN_THREADS / 32);
    for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_windows; w += warps) {
        const int64_t r = akwin_owner(wsplits, A.n_pairs, w, lane), k = w - wsplits[r];
        const int64_t ra = A.splits_a[r] + (A.bos >= 0), rb = A.splits_b[r] + (A.bos >= 0);
        const int s = (A.bos >= 0) + (A.eos >= 0);
        int64_t ca = A.splits_a[r + 1] - A.splits_a[r] - s, cb = A.splits_b[r + 1] - A.splits_b[r] - s;
        ca = ca > 0 ? ca : 0;
        cb = cb > 0 ? cb : 0;
        const AkPairPlan p = akpair_plan(ca, cb, A.m, A.stride, A.strategy, A.overflow);
        int64_t i, j, a0, a1, b0, b1;
        akpair_ij(k, p.wa, p.wb, i, j);
        akwin_span(ca, p.na, p.na - A.stride, A.left, i, a0, a1);
        akwin_span(cb, p.nb, p.nb - A.stride, A.left, j, b0, b1);
        // segment ends in the window: pre | A_i | mid | B_j | post
        const int64_t e0 = A.n_pre, e1 = e0 + (a1 - a0), e2 = e1 + A.n_mid, e3 = e2 + (b1 - b0), total = e3 + A.n_post;
        const int64_t first = A.pad_left ? width - total : 0;    // output position of the window's first id
        const IdT* srca = A.ids_a + ra + a0 - e0;                // srca[p]: the id at window position p, for p in [e0, e1)
        const IdT* srcb = A.ids_b + rb + b0 - e2;
        int64_t* oi = out_ids + w * width;
        int64_t* om = out_mask + w * width;
        for (int64_t j0 = 0; j0 < width; j0 += 32 * AKWIN_UNROLL) {
            int64_t v[AKWIN_UNROLL];
#pragma unroll
            for (int u = 0; u < AKWIN_UNROLL; ++u) {
                const int64_t q = j0 + u * 32 + lane - first;
                const bool in_a = q >= e0 && q < e1, in_b = q >= e2 && q < e3;
                const IdT* src = q < e2 ? srca : srcb;
                const int t = (int)(q < e0 ? q : q < e2 ? AKPAIR_SLOT + (q - e1) : 2 * AKPAIR_SLOT + (q - e3)) & 15;
                v[u] = in_a || in_b ? (int64_t)src[q] : q < 0 || q >= total ? pad_id : (int64_t)s_tmpl[t];
            }
#pragma unroll
            for (int u = 0; u < AKWIN_UNROLL; ++u) {
                const int64_t jj = j0 + u * 32 + lane, q = jj - first;
                if (jj < width) {
                    oi[jj] = v[u];
                    om[jj] = q >= 0 && q < total;
                }
            }
        }
        if (lane == 0) sample[w] = r;
    }
}
