// Kernels of the model-ready windows (ragged ids -> input_ids / attention_mask [N, L], the rule of HF tokenizers'
// truncation with stride + padding; include/akshar_b200.h, akshar_windows_count / akshar_windows_write).
//   ak_win_count_kernel    one thread per row: its window count, the template check, the longest window
//   (ak_scan_counts_kernel) window splits of the rows, N
//   ak_win_write_kernel    one warp per window: its row by a 32-way search in the window splits, then the L positions of
//                          both outputs as coalesced int64 stores
// The write is a gather: ids are read once per window position they land in, 16 bytes are written per output position.
#pragma once
#include "ak_win.cuh"

#define AKWIN_THREADS 256

template <class IdT>
struct AkWinArgs {
    const IdT* ids;
    const int64_t* splits;             // [n_rows + 1] positions in ids
    int64_t n_rows;
    int32_t bos, eos;                  // template ids, -1: none
    int64_t m;                         // content ids per window (max_length - template ids); truncation off: INT64_MAX
    int64_t step;                      // m - stride
    bool overflow, left, pad_left;
};

// count[r] = windows of row r (count[n_rows] = 0, so that the scan's last entry is N); result[1] = longest window;
// AKSHAR_ST_TEMPLATE when a row is not framed by the template ids
template <class IdT>
__global__ void __launch_bounds__(AKWIN_THREADS) ak_win_count_kernel(const AkWinArgs<IdT> A, int32_t* count, int64_t* result) {
    const int s = (A.bos >= 0) + (A.eos >= 0);
    unsigned long long longest = 0;
    uint32_t st = 0;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= A.n_rows; r += (int64_t)gridDim.x * blockDim.x) {
        if (r == A.n_rows) {
            count[r] = 0;
            continue;
        }
        const int64_t lo = A.splits[r], hi = A.splits[r + 1], n = hi - lo;
        if (n < s || (A.bos >= 0 && (int32_t)A.ids[lo] != A.bos) || (A.eos >= 0 && (int32_t)A.ids[hi - 1] != A.eos)) st |= AKSHAR_ST_TEMPLATE;
        const int64_t c = n > s ? n - s : 0;
        int64_t w = 1;
        if (c > A.m && A.overflow) w = 1 + (c - A.m + A.step - 1) / A.step;
        count[r] = (int32_t)w;
        const unsigned long long len = (unsigned long long)((c < A.m ? c : A.m) + s);
        longest = len > longest ? len : longest;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, longest, d);
        longest = o > longest ? o : longest;
        st |= __shfl_xor_sync(0xFFFFFFFFu, st, d);
    }
    if ((threadIdx.x & 31) == 0) {
        if (longest) atomicMax((unsigned long long*)&result[1], longest);
        if (st) atomicOr((unsigned int*)&result[2], st);
    }
}

// the row that owns window w, by the whole warp: the last r with wsplits[r] <= w (every row owns at least one window, so
// the window splits increase strictly).  Lane i probes lo + 1 + i (hi - lo) / 32; the probes that pass form a prefix of
// the lanes, so every step divides the range by 32
__device__ __forceinline__ int64_t akwin_owner(const int64_t* __restrict__ wsplits, int64_t n_rows, int64_t w, int lane) {
    int64_t lo = 0, hi = n_rows - 1;
    while (lo < hi) {
        const int64_t q = lo + 1 + ((hi - lo) * lane >> 5);
        const unsigned pass = __ballot_sync(0xFFFFFFFFu, q <= hi && __ldg(wsplits + q) <= w);
        const int last = 31 - __clz(pass | 1u);
        const int64_t q_last = __shfl_sync(0xFFFFFFFFu, q, last), q_next = __shfl_sync(0xFFFFFFFFu, q, last < 31 ? last + 1 : 31);
        if (!pass) hi = lo;
        else {
            hi = last < 31 ? q_next - 1 : hi;
            lo = q_last;
        }
    }
    return lo;
}

// one warp per window: the loads of AKWIN_UNROLL positions are issued before their stores (a load-store chain per
// position leaves the warp waiting on every id), and the owning row is found by a 32-way search (log32 steps)
#define AKWIN_UNROLL 8
template <class IdT>
__global__ void __launch_bounds__(AKWIN_THREADS) ak_win_write_kernel(const AkWinArgs<IdT> A, const int64_t* __restrict__ wsplits, int64_t n_windows,
                                                                     int64_t width, int64_t pad_id, int64_t* __restrict__ out_ids,
                                                                     int64_t* __restrict__ out_mask, int64_t* __restrict__ sample) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (AKWIN_THREADS / 32);
    const int head = A.bos >= 0, s = head + (A.eos >= 0);
    for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_windows; w += warps) {
        const int64_t r = akwin_owner(wsplits, A.n_rows, w, lane), k = w - wsplits[r];
        const int64_t r0 = A.splits[r], n = A.splits[r + 1] - r0;
        const int64_t c = n > s ? n - s : 0;
        int64_t start, stop;
        akwin_span(c, A.m, A.step, A.left, k, start, stop);
        const int64_t len = stop - start, total = len + s;
        const int64_t first = A.pad_left ? width - total : 0;    // output position of the window's first id
        const IdT* src = A.ids + r0 + start;                     // src[p]: the id at window position p, for p in [head, head + len)
        int64_t* oi = out_ids + w * width;
        int64_t* om = out_mask + w * width;
        for (int64_t j0 = 0; j0 < width; j0 += 32 * AKWIN_UNROLL) {
            int64_t v[AKWIN_UNROLL];
#pragma unroll
            for (int u = 0; u < AKWIN_UNROLL; ++u) {
                const int64_t p = j0 + u * 32 + lane - first;
                v[u] = p < 0 || p >= total ? pad_id : p < head ? (int64_t)A.bos : p < head + len ? (int64_t)src[p] : (int64_t)A.eos;
            }
#pragma unroll
            for (int u = 0; u < AKWIN_UNROLL; ++u) {
                const int64_t j = j0 + u * 32 + lane, p = j - first;
                if (j < width) {
                    oi[j] = v[u];
                    om[j] = p >= 0 && p < total;
                }
            }
        }
        if (lane == 0) sample[w] = r;
    }
}
