// Compiles the n-tuple arithmetic of the PRODUCT's device header (ml2048_b200/csrc/board_ops.cuh) as plain C++, so that the
// symmetry maps, the index and the value can be checked against the NumPy reference without a GPU.
// Test infrastructure only (tests/test_ntuple_ref.py).
#include <stdint.h>
#include <string.h>

#include "../../ml2048_b200/csrc/board_ops.cuh"

using namespace ml2048;

extern "C" {

uint32_t nt_sym_src(uint32_t g, uint32_t cell) { return ntuple_sym_src(g, cell); }

// expand cells [K][6] + len [K]: returns the entry count, copies offsets [K] and src4 [K][8][8]
int64_t nt_expand(const uint8_t *cells, const uint8_t *len, int32_t k, uint32_t *offsets, uint8_t *src4)
{
    NTupleSpec s;
    const int64_t n = ntuple_expand(cells, len, k, s);
    memcpy(offsets, s.offset, 4 * (size_t)k);
    memcpy(src4, s.src4, 64 * (size_t)k);
    return n;
}

// index of tuple t, image g for n boards
void nt_index_batch(const uint8_t *boards, int64_t n, const uint8_t *cells, const uint8_t *len, int32_t k, int32_t t, int32_t g,
                    uint32_t *out)
{
    NTupleSpec s;
    ntuple_expand(cells, len, k, s);
    for (int64_t i = 0; i < n; ++i) {
        uint32_t r[4];
        memcpy(r, boards + 16 * i, 16);
        out[i] = ntuple_index(ntuple_nibbles(r[0], r[1], r[2], r[3]), s.src4[t][g], s.len[t]);
    }
}

void nt_value_batch(const uint8_t *boards, int64_t n, const float *w, const uint8_t *cells, const uint8_t *len, int32_t k, float *out)
{
    NTupleSpec s;
    ntuple_expand(cells, len, k, s);
    for (int64_t i = 0; i < n; ++i) {
        uint32_t r[4];
        memcpy(r, boards + 16 * i, 16);
        out[i] = ntuple_value(w, s, ntuple_nibbles(r[0], r[1], r[2], r[3]));
    }
}

}  // extern "C"
