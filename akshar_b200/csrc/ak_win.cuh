// Window arithmetic of the model-ready batches (include/akshar_b200.h, akshar_windows_count and
// akshar_pair_windows_count): where a window of a row lies in its content, and how HF tokenizers 0.22.2 cuts a
// sentence pair (truncate_encodings + Encoding::truncate + Encoding::merge_with).  AK_HD so that the CPU tests can
// check it against the plain-Python rule (tools/windows_oracle.py) without a GPU.
#pragma once
#include <stdint.h>
#include "ak_unicode.cuh"

// window k of a row with c content ids, cut to windows of m ids that step by `step`: [start, stop) in the content
AK_HD void akwin_span(int64_t c, int64_t m, int64_t step, bool left, int64_t k, int64_t& start, int64_t& stop) {
    if (c <= m) {
        start = 0;
        stop = c;
    } else if (left) {
        stop = c - k * step;
        start = stop > m ? stop - m : 0;
    } else {
        start = k * step;
        stop = start + m < c ? start + m : c;
    }
}

// truncation strategy of a pair (AKSHAR_WIN_TRUNCATE + AKSHAR_WIN_ONLY_FIRST / AKSHAR_WIN_ONLY_SECOND)
enum { AKPAIR_NONE = 0, AKPAIR_LONGEST_FIRST = 1, AKPAIR_ONLY_FIRST = 2, AKPAIR_ONLY_SECOND = 3 };
// why a pair is refused (HF misbehaves or raises there)
enum {
    AKPAIR_OK = 0,
    AKPAIR_CUT_TO_ZERO = 1,   // longest_first would cut a sequence to 0 ids (HF returns windows wider than max_length)
    AKPAIR_STRIDE = 2,        // stride >= the length a sequence is cut to (HF panics)
    AKPAIR_TOO_SHORT = 3,     // only_first / only_second: the sequence to cut has no more ids than must go (HF raises)
    AKPAIR_TOO_MANY = 4,      // more than 2^31 - 1 windows
    AKPAIR_CALL_TOO_MANY = 5, // (the whole call, not one pair) more than 2^31 - 1 windows in all
};

struct AkPairPlan {
    int64_t na, nb;           // the lengths A and B are cut to (their own length when not cut)
    int64_t wa, wb;           // windows of A and of B: the pair has wa * wb windows
    int reason;               // AKPAIR_OK or why the pair is refused
};

// windows of a sequence of c ids cut to n (n < c) with `stride`: 1 + ceil((c - n) / (n - stride)); 1 when not cut.
// Every length is below 2^31 (the ids of one call), so the division is a 32-bit one
AK_HD int64_t akpair_windows(int64_t c, int64_t n, int64_t stride, bool overflow) {
    if (c <= n || !overflow) return 1;
    const uint32_t step = (uint32_t)(n - stride);
    return 1 + (int64_t)(((uint32_t)(c - n) + step - 1) / step);
}

// the plan of a pair with contents of ca and cb ids, m = max_length - the pair template's ids (> 0)
AK_HD AkPairPlan akpair_plan(int64_t ca, int64_t cb, int64_t m, int64_t stride, int strategy, bool overflow) {
    AkPairPlan P;
    P.na = ca;
    P.nb = cb;
    P.wa = P.wb = 1;
    P.reason = AKPAIR_OK;
    if (strategy == AKPAIR_NONE || ca + cb <= m) return P;
    if (strategy == AKPAIR_LONGEST_FIRST) {
        const bool swap = ca > cb;
        int64_t n1 = swap ? cb : ca, n2;
        if (n1 > m) n2 = n1;
        else n2 = n1 > m - n1 ? n1 : m - n1;
        if (n1 + n2 > m) {
            n1 = m >> 1;
            n2 = n1 + (m & 1);
        }
        P.na = swap ? n2 : n1;
        P.nb = swap ? n1 : n2;
        if (P.na > ca) P.na = ca;     // a sequence is never lengthened: n >= len leaves it whole
        if (P.nb > cb) P.nb = cb;
    } else {
        const int64_t rem = ca + cb - m;
        const int64_t len = strategy == AKPAIR_ONLY_FIRST ? ca : cb;
        if (len <= rem) {
            P.reason = AKPAIR_TOO_SHORT;
            return P;
        }
        if (strategy == AKPAIR_ONLY_FIRST) P.na = ca - rem;
        else P.nb = cb - rem;
    }
    if ((P.na < ca && P.na == 0) || (P.nb < cb && P.nb == 0)) {
        P.reason = AKPAIR_CUT_TO_ZERO;
        return P;
    }
    if ((P.na < ca && stride >= P.na) || (P.nb < cb && stride >= P.nb)) {
        P.reason = AKPAIR_STRIDE;
        return P;
    }
    P.wa = akpair_windows(ca, P.na, stride, overflow);
    P.wb = akpair_windows(cb, P.nb, stride, overflow);
    if (P.wa * P.wb > INT32_MAX) P.reason = AKPAIR_TOO_MANY;
    return P;
}

// window k of a pair -> (window i of A, window j of B) in merge_with's order: (0, 0); (i, 0 .. wb - 1) for
// i = 1 .. wa - 1; then (0, j) for j = 1 .. wb - 1.  k < wa * wb < 2^31: 32-bit division
AK_HD void akpair_ij(int64_t k, int64_t wa, int64_t wb, int64_t& i, int64_t& j) {
    if (k == 0) {
        i = j = 0;
    } else if (k <= (wa - 1) * wb) {
        const uint32_t q = (uint32_t)(k - 1) / (uint32_t)wb;
        i = 1 + (int64_t)q;
        j = (k - 1) - (int64_t)q * wb;
    } else {
        i = 0;
        j = k - (wa - 1) * wb;
    }
}
