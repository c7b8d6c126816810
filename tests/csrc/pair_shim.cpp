// CPU build of the sentence-pair window arithmetic (akshar_b200/csrc/ak_win.cuh) and of the pair-template loader, for
// tests/test_pair_windows.py (test aid only: the product runs the CUDA build of the same header).
#include <stdint.h>
#include <string>

#include "../../akshar_b200/csrc/ak_models.h"
#include "../../akshar_b200/csrc/ak_win.cuh"

extern "C" {

// the windows of one pair as the write kernel computes them: out[4 k ..] = startA, stopA, startB, stopB of window k;
// returns the number of windows, or -reason when the pair is refused
int64_t ps_pair_windows(int64_t ca, int64_t cb, int64_t m, int64_t stride, int strategy, int left, int overflow, int64_t* out,
                        int64_t cap) {
    const AkPairPlan p = akpair_plan(ca, cb, m, stride, strategy, overflow != 0);
    if (p.reason) return -p.reason;
    const int64_t n = p.wa * p.wb;
    for (int64_t k = 0; k < n && k < cap; ++k) {
        int64_t i, j;
        akpair_ij(k, p.wa, p.wb, i, j);
        akwin_span(ca, p.na, p.na - stride, left != 0, i, out[4 * k], out[4 * k + 1]);
        akwin_span(cb, p.nb, p.nb - stride, left != 0, j, out[4 * k + 2], out[4 * k + 3]);
    }
    return n;
}

// the pair slots of a tokenizer JSON: returns 1 when the pair template is usable, 0 when not, -1 when the model does
// not load; n[3] ids per slot, ids[3][4]
int ps_load_pair(const char* json, int64_t len, int32_t* n, int32_t* ids) {
    AkBpeHost h;
    if (!ak_parse_bpe_json(json, (size_t)len, h).empty()) return -1;
    for (int s = 0; s < 3; ++s) {
        n[s] = h.pair_n[s];
        for (int i = 0; i < 4; ++i) ids[4 * s + i] = h.pair_ids[s][i];
    }
    return h.pair_ok ? 1 : 0;
}
}
