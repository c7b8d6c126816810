// CPU build of the word cache (akshar_b200/csrc/ak_wordcache.cuh), for tests/test_word_cache.py (test aid only: the
// product runs the CUDA build of the same header).  A table is the caller's array of (1 << bits) x AKC_ENTRY u64.
#include <stdint.h>

#include "../../akshar_b200/csrc/ak_wordcache.cuh"

static AkWordCache wc_table(unsigned long long* e, uint32_t bits, unsigned long long* inserted) {
    AkWordCache C;
    C.e = e;
    C.bits = bits;
    C.inserted = inserted;
    return C;
}

extern "C" {

// look the word [t, t + len) up: out = {hash, slot, free_slot}
void wc_lookup(unsigned long long* e, uint32_t bits, const uint8_t* t, uint32_t len, int64_t* out) {
    const AkWordCache C = wc_table(e, bits, nullptr);
    unsigned long long k[4];
    akc_key0123(t, 0, len, (int64_t)len, k);
    AkcHit r;
    akc_lookup4(C, t, 0, len, k, r);
    out[0] = (int64_t)r.h;
    out[1] = r.slot;
    out[2] = r.free_slot;
}

// the hash akc_lookup4 computes for each of n words (word i = bytes [off[i], off[i + 1]) of t)
void wc_hash(const uint8_t* t, const int64_t* off, int64_t n, uint64_t* out) {
    unsigned long long empty[AKC_ENTRY] = {0};
    for (int64_t i = 0; i < n; ++i) {
        int64_t r[3];
        wc_lookup(empty, 0, t + off[i], (uint32_t)(off[i + 1] - off[i]), r);
        out[i] = (uint64_t)r[0];
    }
}

// a miss with a free slot on the probe path is published there, as the encoders publish a word; returns the slot, or
// -1 when the word was found or found no free slot
int64_t wc_insert(unsigned long long* e, uint32_t bits, const uint8_t* t, uint32_t len, const int32_t* ids, int n,
                  unsigned long long* inserted) {
    const AkWordCache C = wc_table(e, bits, inserted);
    unsigned long long k[4];
    akc_key0123(t, 0, len, (int64_t)len, k);
    AkcHit r;
    akc_lookup4(C, t, 0, len, k, r);
    if (r.slot >= 0 || r.free_slot < 0) return -1;
    akc_insert(C, r.free_slot, r.want, t, 0, len, ids, n, 0ull);
    return r.free_slot;
}

// the ids of a hit, as the encoders read them (the first two from the tag's sector, the others with akc_id);
// returns their count, -1 on a miss
int wc_get(unsigned long long* e, uint32_t bits, const uint8_t* t, uint32_t len, int32_t* ids) {
    const AkWordCache C = wc_table(e, bits, nullptr);
    unsigned long long k[4];
    akc_key0123(t, 0, len, (int64_t)len, k);
    AkcHit r;
    akc_lookup4(C, t, 0, len, k, r);
    if (r.slot < 0) return -1;
    const int n = AKC_NTOK(r.tag);
    for (int i = 0; i < n; ++i)
        ids[i] = i < 2 ? (int32_t)(uint32_t)(r.ids01 >> (32 * i)) : (int32_t)akc_id(C.e + r.slot * AKC_ENTRY, i);
    return n;
}
}
