// Compiles the stage arithmetic of the PRODUCT's device header (ml2048_b200/csrc/board_ops.cuh) as plain C++, so that the
// stage table, the stage of a board and the staged value can be checked against the NumPy reference without a GPU.
// Test infrastructure only (tests/test_stages_ref.py).
#include <stdint.h>
#include <string.h>

#include "../../ml2048_b200/csrc/board_ops.cuh"

using namespace ml2048;

extern "C" {

uint64_t st_table(const uint8_t *tau, int32_t num_stages) { return ntuple_stage_table(tau, num_stages); }

// stage of n boards under thresholds tau [S-1]
void st_stage_batch(const uint8_t *boards, int64_t n, const uint8_t *tau, int32_t num_stages, uint32_t *out)
{
    NTupleStagedSpec s{};
    s.stage_of = ntuple_stage_table(tau, num_stages);
    for (int64_t i = 0; i < n; ++i) {
        uint32_t r[4];
        memcpy(r, boards + 16 * i, 16);
        out[i] = ntuple_stage(s, ntuple_nibbles(r[0], r[1], r[2], r[3]));
    }
}

// staged value of n boards: tuples cells [K][6] + len [K], weights [S * N]
void st_value_batch(const uint8_t *boards, int64_t n, const float *w, const uint8_t *cells, const uint8_t *len, int32_t k,
                    const uint8_t *tau, int32_t num_stages, float *out)
{
    NTupleStagedSpec s{};
    s.stage_size = (uint32_t)ntuple_expand(cells, len, k, s);
    s.stage_of = ntuple_stage_table(tau, num_stages);
    for (int64_t i = 0; i < n; ++i) {
        uint32_t r[4];
        memcpy(r, boards + 16 * i, 16);
        out[i] = ntuple_value(w, s, ntuple_nibbles(r[0], r[1], r[2], r[3]));
    }
}

}  // extern "C"
