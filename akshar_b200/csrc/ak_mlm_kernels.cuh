// Kernel of the masked language-model batches (DataCollatorForLanguageModeling(mlm=True)'s 80/10/10 masking of a dense
// [N, L] batch in place; include/akshar_b200.h, akshar_mlm_mask).
//   ak_mlm_kernel   elementwise, grid-stride over pairs of positions: one 16-byte load of two ids, a Philox block and the
//                   rule of ak_mlm.cuh per position, one 16-byte store of two labels, an 8-byte store per changed id
// No workspace, no scan, no read-back.  Per position: 8 bytes read, 8 written, and the changed ids (about 13.5 % at the
// default probabilities) scattered.
#pragma once
#include "ak_mlm.cuh"

#define AKMLM_THREADS 256

struct AkMlmArgs {
    int64_t* ids;                      // [N L], changed in place
    int64_t* labels;                   // [N L]
    int64_t total;                     // N L
    int64_t L;                         // width, < 2^32
    int64_t d_row, d_col;              // the grid's stride in positions (2 per thread) as whole rows and columns
    uint64_t row_base;
    uint64_t t[3];                     // thresholds, each <= 2^32
    uint32_t key[2];                   // the seed's two words
    uint32_t epoch;
    uint32_t V;                        // ids drawn at random are in [0, V)
    int64_t mask_id;
    int64_t pad_id;                    // -1: none
    const uint32_t* special;           // one bit per id of the model's special ids
    int64_t n_bits;
    int vec;                           // ids and labels 16-byte aligned: pairs are moved as one 16-byte access
};

// the position (row, col) holding `id`: its new id, and its label in *label
__device__ __forceinline__ int64_t akmlm_at(const AkMlmArgs& A, int64_t id, int64_t row, int64_t col, int64_t* label) {
    const uint64_t R = A.row_base + (uint64_t)row;
    const uint32_t c[4] = {(uint32_t)col, (uint32_t)R, (uint32_t)(R >> 32), A.epoch};
    uint32_t u[4];
    akmlm_philox(c, A.key, u);
    const bool special = (A.pad_id >= 0 && id == A.pad_id) ||
                         ((uint64_t)id < (uint64_t)A.n_bits && ((__ldg(A.special + (id >> 5)) >> (id & 31)) & 1u));
    return akmlm_position(id, special, u, A.t, A.mask_id, A.V, label);
}

__global__ void __launch_bounds__(AKMLM_THREADS) ak_mlm_kernel(const AkMlmArgs A) {
    const int64_t n_pairs = (A.total + 1) >> 1, stride = (int64_t)gridDim.x * blockDim.x;
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_pairs) return;
    int64_t row = 2 * k / A.L, col = 2 * k - row * A.L;       // the one division of the thread; then it only adds
    for (; k < n_pairs; k += stride) {
        const int64_t i = 2 * k;
        const bool two = i + 1 < A.total;
        int64_t a, b = 0;
        if (A.vec && two) {
            const longlong2 v = __ldcs((const longlong2*)(A.ids + i));
            a = v.x;
            b = v.y;
        } else {
            a = A.ids[i];
            if (two) b = A.ids[i + 1];
        }
        int64_t la, lb = -100;
        const int64_t na = akmlm_at(A, a, row, col, &la);
        int64_t nb = b;
        if (two) nb = col + 1 < A.L ? akmlm_at(A, b, row, col + 1, &lb) : akmlm_at(A, b, row + 1, 0, &lb);
        if (A.vec && two) {
            __stcs((longlong2*)(A.labels + i), make_longlong2(la, lb));
        } else {
            A.labels[i] = la;
            if (two) A.labels[i + 1] = lb;
        }
        if (na != a) A.ids[i] = na;
        if (two && nb != b) A.ids[i + 1] = nb;
        col += A.d_col;
        row += A.d_row;
        if (col >= A.L) {
            col -= A.L;
            ++row;
        }
    }
}
