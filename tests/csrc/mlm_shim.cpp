// CPU build of the masked-LM arithmetic (akshar_b200/csrc/ak_mlm.cuh), for tests/test_mlm.py (test aid only: the product
// runs the CUDA build of the same header).
#include <stdint.h>

#include "../../akshar_b200/csrc/ak_mlm.cuh"

extern "C" {

// n Philox blocks: ctr [4 n], key [2 n] -> out [4 n]
void ms_philox(const uint32_t* ctr, const uint32_t* key, int64_t n, uint32_t* out) {
    for (int64_t i = 0; i < n; ++i) akmlm_philox(ctr + 4 * i, key + 2 * i, out + 4 * i);
}

// an [n_rows, width] batch as the kernel masks it (is_special [n_ids]: 1 for a special id): ids in place, labels
void ms_mask(int64_t* ids, int64_t n_rows, int64_t width, uint64_t seed, uint32_t epoch, uint64_t row_base, const uint64_t* t,
             int64_t mask_id, int64_t pad_id, uint32_t V, const uint8_t* is_special, int64_t n_ids, int64_t* labels) {
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    for (int64_t n = 0; n < n_rows; ++n) {
        const uint64_t R = row_base + (uint64_t)n;
        for (int64_t j = 0; j < width; ++j) {
            const uint32_t c[4] = {(uint32_t)j, (uint32_t)R, (uint32_t)(R >> 32), epoch};
            uint32_t u[4];
            akmlm_philox(c, key, u);
            int64_t& id = ids[n * width + j];
            const bool special = (pad_id >= 0 && id == pad_id) || (id >= 0 && id < n_ids && is_special[id]);
            id = akmlm_position(id, special, u, t, mask_id, V, &labels[n * width + j]);
        }
    }
}
}
