// Compiles the PRODUCT's device header (ml2048_b200/csrc/board_ops.cuh) as plain C++ so that its SWAR
// arithmetic can be checked exhaustively against the CPU oracle on a machine without a GPU.
// Test infrastructure only (tests/test_board_ops_host.py).
#include <stdint.h>
#include <string.h>

#include "../../ml2048_b200/csrc/board_ops.cuh"

using namespace ml2048;

extern "C" {

void hs_move(const uint8_t *board16, int action, uint8_t *out16, uint32_t *gain, uint32_t *rank, uint32_t *count,
             uint8_t *merged16)
{
    uint32_t r[4];
    memcpy(r, board16, 16);
    Fusions f;
    move_board(r[0], r[1], r[2], r[3], (uint32_t)action, f);
    memcpy(out16, r, 16);
    *gain = (uint32_t)fusion_gain(f);
    *rank = fusion_rank(f);
    *count = fusion_count(f);
    uint32_t m[4];
    fusion_log(f, m[0], m[1], m[2], m[3]);
    memcpy(merged16, m, 16);
}

uint32_t hs_valid_mask(const uint8_t *board16)
{
    uint32_t r[4];
    memcpy(r, board16, 16);
    return valid_mask(r[0], r[1], r[2], r[3]);
}

uint32_t hs_first_empty(const uint8_t *keys16, const uint8_t *board16)
{
    uint32_t k[4], r[4];
    memcpy(k, keys16, 16);
    memcpy(r, board16, 16);
    return first_empty_by_rank(k[0], k[1], k[2], k[3], occupied_flags(r[0]), occupied_flags(r[1]), occupied_flags(r[2]),
                               occupied_flags(r[3]));
}

uint32_t hs_max_cell(const uint8_t *board16)
{
    uint32_t r[4];
    memcpy(r, board16, 16);
    return max_cell(r[0], r[1], r[2], r[3]);
}

uint32_t hs_empties16(const uint8_t *board16)
{
    uint32_t r[4];
    memcpy(r, board16, 16);
    return empties16(occupied_flags(r[0]) ^ kHi, occupied_flags(r[1]) ^ kHi, occupied_flags(r[2]) ^ kHi,
                     occupied_flags(r[3]) ^ kHi);
}

uint32_t hs_kth_set_bit16(uint32_t mask, uint32_t k) { return kth_set_bit16(mask, k); }

uint32_t hs_mask_bits4(uint32_t valid_word) { return mask_bits4(valid_word); }

uint32_t hs_kth_valid_action(uint32_t bits, uint32_t k) { return kth_valid_action(bits, k); }

void hs_put_cell(uint8_t *board16, uint32_t cell, uint32_t value)
{
    uint32_t r[4];
    memcpy(r, board16, 16);
    uint32_t q[4] = {r[0], r[1], r[2], r[3]};
    put_cell(r[0], r[1], r[2], r[3], cell, value);
    put_cell_shift(q[0], q[1], q[2], q[3], cell, value);
    if (memcmp(q, r, 16) != 0) r[0] = r[1] = r[2] = r[3] = 0xffffffffu;  // the two forms must agree (the test then fails on the board)
    memcpy(board16, r, 16);
}

void hs_philox(const uint32_t *ctr4, const uint32_t *key2, uint32_t *out4)
{
    const u32x4 o = philox4x32_10(ctr4[0], ctr4[1], ctr4[2], ctr4[3], key2[0], key2[1]);
    out4[0] = o.x, out4[1] = o.y, out4[2] = o.z, out4[3] = o.w;
}

// the (mask, k)-indexed selector table of the in-kernel random policy: copies the 64 rows of 8 words
void hs_policy_sel_table(uint32_t *out512)
{
    static const PolicySelTable t = make_policy_sel_table();
    memcpy(out512, t.w, sizeof(t.w));
}

// the 1024 boards a reset can produce + their masks: copies 1024 x 4 board words and 1024 mask words
void hs_fresh_table(uint32_t *boards4096, uint32_t *masks1024)
{
    static const FreshTable t = make_fresh_table();
    memcpy(boards4096, t.board, sizeof(t.board));
    memcpy(masks1024, t.mask, sizeof(t.mask));
}

void hs_move_sel_table(uint32_t *out32)
{
    static const uint32_t base[4 * kMoveSelRow] = ML2048_MOVE_SEL_TABLE;
    memcpy(out32, base, sizeof(base));
}

void hs_philox2(const uint32_t *ctr2, uint32_t key, uint32_t *out2)
{
    const u32x2 o = philox2x32_10(ctr2[0], ctr2[1], key);
    out2[0] = o.x, out2[1] = o.y;
}

uint32_t hs_slot_word(uint64_t slot, uint64_t counter, uint64_t seed, uint32_t tag) { return slot_word(slot, counter, seed, tag); }

void hs_slot_draws(uint64_t slot, uint64_t counter, uint64_t seed, uint32_t tag, uint32_t *out2)
{
    const u32x2 o = slot_draws(slot, counter, seed, tag);
    out2[0] = o.x, out2[1] = o.y;
}

// batched drivers (keep the Python loops out of the exhaustive tests)
void hs_move_batch(const uint8_t *boards, int64_t n, int action, uint8_t *out, uint32_t *gain, uint32_t *rank, uint32_t *count,
                   uint8_t *merged, uint32_t *mask_before)
{
    for (int64_t i = 0; i < n; ++i) {
        hs_move(boards + 16 * i, action, out + 16 * i, gain + i, rank + i, count + i, merged + 16 * i);
        mask_before[i] = hs_valid_mask(boards + 16 * i);
    }
}

void hs_first_empty_batch(const uint8_t *keys, const uint8_t *boards, int64_t n, uint32_t *cells)
{
    for (int64_t i = 0; i < n; ++i) cells[i] = hs_first_empty(keys + 16 * i, boards + 16 * i);
}

// logits (n,4) f32, bits (n,) = 4-bit valid masks, words (n,) = the policy's uniform words
void hs_sample_masked_categorical_batch(const float *logits, const uint8_t *bits, const uint32_t *words, int64_t n,
                                        uint8_t *actions, float *log_probs)
{
    for (int64_t i = 0; i < n; ++i) {
        const float *l = logits + 4 * i;
        actions[i] = (uint8_t)sample_masked_categorical(l[0], l[1], l[2], l[3], bits[i], words[i], log_probs[i]);
    }
}

}  // extern "C"
