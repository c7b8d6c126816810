// CPU build of the packed-batch arithmetic (akshar_b200/csrc/ak_pack.cuh), for tests/test_packing.py (test aid only:
// the product runs the CUDA build of the same header).
#include <stdint.h>

#include "../../akshar_b200/csrc/ak_pack.cuh"

extern "C" {

// units [starts[u], starts[u + 1]) of a stream of starts[n_units] ids: out[3 u ..] = pieces below NL, longest piece,
// rest fragments
void ps_pack_units(const int64_t* starts, int64_t n_units, int64_t L, int64_t NL, int64_t* out) {
    for (int64_t u = 0; u < n_units; ++u) {
        const AkPackUnit U = akpack_unit(starts[u], starts[u + 1], L, NL);
        out[3 * u] = U.main;
        out[3 * u + 1] = U.longest;
        out[3 * u + 2] = U.rest;
    }
}

// position_ids and seq_idx of positions [0, NL) as the write kernel computes them, with first[u] = the index of unit u's
// first piece (the exclusive prefix sum of the pieces)
void ps_pack_positions(const int64_t* starts, int64_t n_units, const int64_t* first, int64_t L, int64_t NL, int32_t* pos,
                       int32_t* seq) {
    int64_t u = 0;
    for (int64_t p = 0; p < NL; ++p) {
        while (u + 1 < n_units && starts[u + 1] <= p) ++u;
        akpack_position((uint32_t)p, (uint32_t)starts[u], (uint32_t)L, (int32_t)first[u], pos[p], seq[p]);
    }
}

void ps_pack_position(int64_t p, int64_t s, int64_t L, int64_t k, int32_t* pos, int32_t* seq) {
    akpack_position((uint32_t)p, (uint32_t)s, (uint32_t)L, (int32_t)k, *pos, *seq);
}
}
