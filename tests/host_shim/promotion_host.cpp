// Compiles the weight-promotion arithmetic of the PRODUCT's device header (ml2048_b200/csrc/board_ops.cuh) as plain C++, so
// that the source stage and the promoted value can be checked against the NumPy reference without a GPU.
// Test infrastructure only (tests/test_promotion_ref.py).
#include <stdint.h>
#include <string.h>

#include "../../ml2048_b200/csrc/board_ops.cuh"

using namespace ml2048;

extern "C" {

uint32_t pr_source_stage(uint32_t s, uint32_t m) { return ntuple_source_stage(s, m); }

// promoted value of n boards: tuples cells [K][6] + len [K], weights [S * N], marks [N]
void pr_value_batch(const uint8_t *boards, int64_t n, const float *w, const uint8_t *cells, const uint8_t *len, int32_t k,
                    const uint8_t *tau, int32_t num_stages, const uint8_t *promoted, float *out)
{
    NTuplePromotedSpec s{};
    s.stage_size = (uint32_t)ntuple_expand(cells, len, k, s);
    s.stage_of = ntuple_stage_table(tau, num_stages);
    s.promoted = promoted;
    for (int64_t i = 0; i < n; ++i) {
        uint32_t r[4];
        memcpy(r, boards + 16 * i, 16);
        out[i] = ntuple_value(w, s, ntuple_nibbles(r[0], r[1], r[2], r[3]));
    }
}

}  // extern "C"
