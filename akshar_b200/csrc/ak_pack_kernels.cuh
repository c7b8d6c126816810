// Kernels of the packed language-model batches (ragged ids -> fixed blocks of L ids with per-document position_ids,
// labels, seq_idx and cu_seq_lens, the rule of transformers' group_texts + DataCollatorWithFlattening;
// include/akshar_b200.h, akshar_pack_count / akshar_pack_write).
//   ak_pack_count_kernel   one thread per unit (carry fragment or row): its stream start, its pieces and rest fragments
//                          from the closed forms of ak_pack.cuh, the longest piece
//   (ak_scan_counts_kernel) the index of every unit's first piece (rest fragments are numbered after the pieces)
//   ak_pack_write_kernel   one warp per tile of AKPACK_TILE consecutive stream positions: the unit of the first position
//                          by a 32-way search, the units of the others from a window of 32 unit starts held in lanes; then
//                          every output of a position as coalesced stores, the rest (positions >= N L) in stream form
// The ids are read once, in stream order; 28 bytes are written per position with every output asked for.
#pragma once
#include "ak_pack.cuh"

#define AKPACK_THREADS 256
#define AKPACK_UNROLL 8
#define AKPACK_TILE (32 * AKPACK_UNROLL)

template <class IdT>
struct AkPackArgs {
    const IdT* ids;
    const int64_t* splits;             // [n_rows + 1] positions in ids
    int64_t n_rows;
    const int32_t* carry;              // the carry's ids (NULL when it holds none)
    const int64_t* carry_splits;       // [n_carry + 1] positions in carry (NULL when n_carry = 0)
    int64_t n_carry;
    int64_t eos;                       // appended to every row; -1: none
    int64_t L;                         // block size
};

// the stream's extent, from the splits: c0 = position of the carry's first id in `carry`, C carry ids, r0 = position of
// the first row's first id in `ids`, T ids in all
template <class IdT>
__device__ __forceinline__ void akpack_extent(const AkPackArgs<IdT>& A, int64_t& c0, int64_t& C, int64_t& r0, int64_t& T) {
    c0 = A.n_carry ? A.carry_splits[0] : 0;
    C = A.n_carry ? A.carry_splits[A.n_carry] - c0 : 0;
    r0 = A.splits[0];
    T = C + (A.splits[A.n_rows] - r0) + (A.eos >= 0 ? A.n_rows : 0);
}

// count[u] = pieces + rest fragments of unit u (count[units] = 0), key[u] = its stream start (key[units] = T);
// result[0] = N, [1] += pieces, [3] = longest piece, [4] = T, [5] += rest fragments; AKSHAR_ST_PACK_LONG when T >= 2^31
template <class IdT>
__global__ void __launch_bounds__(AKPACK_THREADS) ak_pack_count_kernel(const AkPackArgs<IdT> A, int32_t* count, int32_t* key, int64_t* result) {
    int64_t c0, C, r0, T;
    akpack_extent(A, c0, C, r0, T);
    const int64_t units = A.n_carry + A.n_rows, i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (i0 == 0) {
        result[0] = T / A.L;
        result[4] = T;
    }
    if (T > INT32_MAX) {
        // cu_seq_lens and seq_idx are int32: the call is refused; the scan that follows sums zeros
        for (int64_t u = i0; u <= units; u += stride) count[u] = 0;
        if (i0 == 0) atomicOr((unsigned int*)&result[2], (unsigned int)AKSHAR_ST_PACK_LONG);
        return;
    }
    const int64_t NL = T / A.L * A.L, x = A.eos >= 0;
    unsigned long long longest = 0, pieces = 0, frags = 0;
    for (int64_t u = i0; u <= units; u += stride) {
        if (u == units) {
            count[u] = 0;
            key[u] = (int32_t)T;
            continue;
        }
        int64_t s, e;
        if (u < A.n_carry) {
            s = A.carry_splits[u] - c0;
            e = A.carry_splits[u + 1] - c0;
        } else {
            const int64_t r = u - A.n_carry;
            s = C + (A.splits[r] - r0) + x * r;
            e = C + (A.splits[r + 1] - r0) + x * (r + 1);
        }
        const AkPackUnit U = akpack_unit(s, e, A.L, NL);
        count[u] = (int32_t)(U.main + U.rest);
        key[u] = (int32_t)s;
        longest = (unsigned long long)U.longest > longest ? (unsigned long long)U.longest : longest;
        pieces += (unsigned long long)U.main;
        frags += (unsigned long long)U.rest;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, longest, d);
        longest = o > longest ? o : longest;
        pieces += __shfl_xor_sync(0xFFFFFFFFu, pieces, d);
        frags += __shfl_xor_sync(0xFFFFFFFFu, frags, d);
    }
    if ((threadIdx.x & 31) == 0) {
        if (longest) atomicMax((unsigned long long*)&result[3], longest);
        if (pieces) atomicAdd((unsigned long long*)&result[1], pieces);
        if (frags) atomicAdd((unsigned long long*)&result[5], frags);
    }
}

// the last unit u in [lo, hi] with key[u] <= p, by the whole warp: the 32-way search of akwin_owner over keys that only
// do not decrease (an empty unit starts where the next one does; the last of them is the one that holds p)
__device__ __forceinline__ int64_t akpack_owner(const int32_t* __restrict__ key, int64_t lo, int64_t hi, int32_t p, int lane) {
    while (lo < hi) {
        const int64_t q = lo + 1 + ((hi - lo) * lane >> 5);
        const unsigned pass = __ballot_sync(0xFFFFFFFFu, q <= hi && __ldg(key + q) <= p);
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

// the same by one thread (a position whose unit lies beyond the window: more than 30 units start in 32 positions)
__device__ __forceinline__ int64_t akpack_owner1(const int32_t* __restrict__ key, int64_t lo, int64_t hi, int32_t p) {
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (__ldg(key + mid) <= p) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// one warp per tile of AKPACK_TILE positions.  Lane i holds the start and first-piece index of unit ub + i; a position's
// unit is found in that window by 5 shuffles, and the window moves on when it no longer reaches past a round of 32
// positions.  The id loads of all AKPACK_UNROLL rounds are issued before the first store (DESIGN section 4.8)
template <class IdT>
__global__ void __launch_bounds__(AKPACK_THREADS) ak_pack_write_kernel(const AkPackArgs<IdT> A, const int32_t* __restrict__ key,
                                                                       const int64_t* __restrict__ base, int64_t n_pieces,
                                                                       int64_t n_frags, int64_t sep, int64_t* __restrict__ out_ids,
                                                                       int64_t* __restrict__ labels, int64_t* __restrict__ pos_out,
                                                                       int32_t* __restrict__ seq_out, int32_t* __restrict__ cu,
                                                                       int32_t* __restrict__ rest_ids, int64_t* __restrict__ rest_splits) {
    const int lane = threadIdx.x & 31;
    int64_t c0, C64, r0, T64;
    akpack_extent(A, c0, C64, r0, T64);
    const int32_t T = (int32_t)T64, C = (int32_t)C64;
    const int32_t NL = (int32_t)(T64 / A.L * A.L);
    const uint32_t L = NL ? (uint32_t)A.L : 1u;             // only positions below NL divide by L
    const int64_t units = A.n_carry + A.n_rows;
    const bool has_eos = A.eos >= 0;
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gtid == 0) {
        if (cu) cu[n_pieces] = NL;
        rest_splits[n_frags] = T - NL;
    }
    const int64_t n_tiles = (T64 + AKPACK_TILE - 1) / AKPACK_TILE, warps = (int64_t)gridDim.x * (AKPACK_THREADS / 32);
    for (int64_t t = gtid >> 5; t < n_tiles; t += warps) {
        const int64_t p0 = t * AKPACK_TILE;            // 64-bit: p0 + 255 may pass INT32_MAX
        int64_t ub = akpack_owner(key, 0, units - 1, (int32_t)p0, lane);
        int32_t wk = ub + lane <= units ? __ldg(key + ub + lane) : INT32_MAX;
        int32_t wb = ub + lane <= units ? (int32_t)__ldg(base + ub + lane) : 0;
        int32_t s[AKPACK_UNROLL], e[AKPACK_UNROLL], k[AKPACK_UNROLL];
        int64_t v[AKPACK_UNROLL];
#pragma unroll
        for (int j = 0; j < AKPACK_UNROLL; ++j) {
            const int64_t q = p0 + 32 * j, p = q + lane;
            s[j] = e[j] = k[j] = 0;
            v[j] = 0;
            if (q >= T) continue;                              // the same for the whole warp
            if (__shfl_sync(0xFFFFFFFFu, wk, 31) <= q + 31) {
                // the window ends inside this round: start it at the unit of the round's first position
                ub = akpack_owner(key, ub, units - 1, (int32_t)q, lane);
                wk = ub + lane <= units ? __ldg(key + ub + lane) : INT32_MAX;
                wb = ub + lane <= units ? (int32_t)__ldg(base + ub + lane) : 0;
            }
            int c = 0;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                const int32_t y = __shfl_sync(0xFFFFFFFFu, wk, c + d);
                if (y <= p) c += d;
            }
            s[j] = __shfl_sync(0xFFFFFFFFu, wk, c);
            e[j] = __shfl_sync(0xFFFFFFFFu, wk, c < 31 ? c + 1 : 31);
            k[j] = __shfl_sync(0xFFFFFFFFu, wb, c);
            if (p >= T) continue;
            int64_t u = ub + c;
            if (c == 31) {
                u = akpack_owner1(key, ub + 31, units - 1, (int32_t)p);
                s[j] = __ldg(key + u);
                e[j] = __ldg(key + u + 1);
                k[j] = (int32_t)__ldg(base + u);
            }
            if (p < C) v[j] = __ldg(A.carry + c0 + p);
            else if (has_eos && p == e[j] - 1) v[j] = A.eos;
            else v[j] = (int64_t)A.ids[r0 + (p - C) - (has_eos ? u - A.n_carry : 0)];
        }
#pragma unroll
        for (int j = 0; j < AKPACK_UNROLL; ++j) {
            const int64_t p = p0 + 32 * j + lane;
            if (p < NL) {
                int32_t pos, seq;
                akpack_position((uint32_t)p, (uint32_t)s[j], L, k[j], pos, seq);
                out_ids[p] = v[j];
                labels[p] = pos ? v[j] : sep;
                if (pos_out) pos_out[p] = pos;
                if (seq_out) seq_out[p] = seq;
                if (cu && pos == 0) cu[seq] = (int32_t)p;
            } else if (p < T) {
                rest_ids[p - NL] = (int32_t)v[j];
                if (p == NL || p == s[j]) {
                    // the unit's rest fragment comes after its pieces: its index among the rest's fragments
                    const AkPackUnit U = akpack_unit(s[j], e[j], A.L, NL);
                    rest_splits[k[j] + U.main - n_pieces] = p - NL;
                }
            }
        }
    }
}
