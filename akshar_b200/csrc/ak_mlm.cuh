// Arithmetic of the masked language-model batches (include/akshar_b200.h, akshar_mlm_mask): the Philox4x32-10 block of a
// position and the collator's 80/10/10 rule applied to it.  AK_HD so that the CPU tests can check it against the
// plain-Python rule (tools/mlm_oracle.py) without a GPU.
#pragma once
#include <stdint.h>
#include "ak_unicode.cuh"

// Philox4x32-10 (Random123, as cuRAND's Philox): out = the block of counter ctr under key
AK_HD void akmlm_philox(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c0 = n0;
        c1 = (uint32_t)p1;
        c2 = n2;
        c3 = (uint32_t)p0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0;
    out[1] = c1;
    out[2] = c2;
    out[3] = c3;
}

// one position: u = (u_select, u_mask, u_random, r_id) of its Philox block, t = the three thresholds (<= 2^32; u < t is
// "drawn").  Returns the new id; *label = the original id where the position is selected, else -100
AK_HD int64_t akmlm_position(int64_t id, bool special, const uint32_t u[4], const uint64_t t[3], int64_t mask_id, uint32_t V,
                             int64_t* label) {
    const bool selected = !special && u[0] < t[0];
    const bool replaced = selected && u[1] < t[1];
    const bool random = selected && !replaced && u[2] < t[2];
    *label = selected ? id : -100;
    return replaced ? mask_id : random ? (int64_t)(((uint64_t)u[3] * V) >> 32) : id;
}
