// Arithmetic of the packed language-model batches (include/akshar_b200.h, akshar_pack_count / akshar_pack_write): the
// pieces a unit of the stream (a carry fragment, or a row with its eos) contributes, and where a position lies in its
// piece.  AK_HD so that the CPU tests can check it against the plain-Python rule (tools/pack_oracle.py) without a GPU.
#pragma once
#include <stdint.h>
#include "ak_unicode.cuh"

struct AkPackUnit {
    int64_t main;      // pieces that start in the unit below NL
    int64_t longest;   // the longest of them (0 without any)
    int64_t rest;      // fragments of the rest that start in it (1 when the unit reaches past NL, else 0)
};

// the unit [s, e) of the stream, blocks of L ids, NL = N L: pieces start at s and at every multiple of L in (s, min(e, NL))
AK_HD AkPackUnit akpack_unit(int64_t s, int64_t e, int64_t L, int64_t NL) {
    AkPackUnit U;
    U.main = U.longest = U.rest = 0;
    if (e <= s) return U;
    U.rest = e > NL;
    if (s >= NL) return U;
    const int64_t m = e < NL ? e : NL;
    const int64_t b0 = s / L, b1 = (m - 1) / L;        // blocks of the unit's first and last position below NL
    U.main = 1 + b1 - b0;
    const int64_t first = ((b0 + 1) * L < m ? (b0 + 1) * L : m) - s;
    U.longest = first;
    if (U.main >= 2) {
        const int64_t last = m - b1 * L;
        U.longest = last > U.longest ? last : U.longest;
    }
    if (U.main >= 3) U.longest = L;
    return U;
}

// position p < NL of the unit that starts at s and whose first piece is piece k: position_ids[p] and seq_idx[p].
// Every position of a call is below 2^31, so the arithmetic is 32-bit
AK_HD void akpack_position(uint32_t p, uint32_t s, uint32_t L, int32_t k, int32_t& pos, int32_t& seq) {
    const uint32_t b = p / L, bl = b * L;
    pos = (int32_t)(p - (s > bl ? s : bl));
    seq = k + (int32_t)(b - s / L);
}
