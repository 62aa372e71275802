// vecgame_kernels.cu -- sm_100a kernels + C ABI for the VecGame hot path (see include/ml2048_b200.h).
//
// Layout in HBM (struct-of-arrays, one entry per game, all owned by the caller):
//   board[2]   uint4   ping-pong: step reads one, writes the other => prev_state costs nothing
//   valid[2]   uint32  ping-pong (left,right,up,down bytes)       => prev_valid_actions costs nothing
//   step i32, score f32, reward f32, terminated u8, invalid u8, id i32, merged uint4 (optional)
// One thread owns one game; a warp's 32 games are contiguous in every array, so every load/store is a
// fully coalesced 32 B..512 B access.  The fused one-hot observation (1 KiB per game in fp32) is
// written cooperatively by the whole block from boards staged in shared memory so that each warp
// store instruction covers 512 contiguous bytes.
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>
#include <utility>

#include "../../include/ml2048_b200.h"
#include "board_ops.cuh"

using namespace ml2048;
namespace cg = cooperative_groups;

namespace {

#ifndef ML2048_STEP_THREADS
#define ML2048_STEP_THREADS 256
#endif
constexpr int kStepThreads = ML2048_STEP_THREADS;   // games per block in the core-only step kernel and the small stand-alone ops
// With a fused one-hot the kernel is a pure HBM write stream; larger blocks (each writing one contiguous
// 768 KiB tile in fp32) measured 3.5 % faster than 256-thread blocks (2844 vs 2949 us at M = 2^24).
#ifndef ML2048_ONEHOT_STEP_THREADS
#define ML2048_ONEHOT_STEP_THREADS 768
#endif
constexpr int kOneHotStepThreads = ML2048_ONEHOT_STEP_THREADS;
#ifndef ML2048_ONEHOT_STEP_MIN_BLOCKS
#define ML2048_ONEHOT_STEP_MIN_BLOCKS 2
#endif
constexpr int kOneHotStepMinBlocks = ML2048_ONEHOT_STEP_MIN_BLOCKS;  // resident blocks per SM the large-batch kernel is compiled for
// Small batches with a fused one-hot (the training shape, M = 2048..4096) are latency-bound: smaller blocks spread the
// one-hot rows over more SMs.
#ifndef ML2048_SMALL_STEP_THREADS
#define ML2048_SMALL_STEP_THREADS 64
#endif
constexpr int kSmallStepThreads = ML2048_SMALL_STEP_THREADS;
// (measured as a fused 16-step graph, fp32 / u8 one-hot, 64- against 256-thread blocks: M = 2^16 15.6 / 8.6 against 16.8 / 9.3 us,
// 2^17 31.8 / 12.4 against 32.2 / 13.0 us, 2^18 55.5 / 18.3 against 56.3 / 19.3 us)
#ifndef ML2048_SMALL_STEP_MAX_GAMES
#define ML2048_SMALL_STEP_MAX_GAMES 131072
#endif
constexpr int64_t kSmallStepMaxGames = ML2048_SMALL_STEP_MAX_GAMES;
constexpr int kPrepThreads = 256;   // threads per block in the auto-reset kernels
constexpr int kPrepTile = kPrepThreads * 16;  // games per block there (16 terminated flags per thread)
constexpr int kRandRows = 1024;     // VecGame._RAND_SIZE, game_numba.py:533

// ---- streaming access helpers ---------------------------------------------------------------

// One-hot tile stores.  Plain st.global measured 2.4 % faster than st.global.cs (evict-first) and the same as
// st.global.wt on B200 for this write stream (2945 vs 3015 us per launch at M = 2^24, fp32), so no cache hint is used.
#if defined(ML2048_STORE_CS)
__device__ __forceinline__ void store_streaming(float4 *p, float4 v) { __stcs(p, v); }
__device__ __forceinline__ void store_streaming(uint4 *p, uint4 v) { __stcs(p, v); }
#else
__device__ __forceinline__ void store_streaming(float4 *p, float4 v) { *p = v; }
__device__ __forceinline__ void store_streaming(uint4 *p, uint4 v) { *p = v; }
#endif

// ---- one-hot tile writer --------------------------------------------------------------------
// out[g][k][c] = (board[g][c] == k) for k < 16 (policy/_network.py:86-95: one_hot(x,16).float().permute(0,2,1)).
// The block's boards sit in shared memory; thread t owns the fixed (class k, column group q) pair
// t mod 64 and walks the games, so one warp instruction stores 32 consecutive 16-byte pieces.

template <int kDtype>
struct OneHotPiece;

template <>
struct OneHotPiece<ML2048_ONEHOT_F32> {  // 4 cells -> 4 floats = 16 bytes; 64 pieces per game
    using vec = float4;
    static constexpr int kPiecesPerGame = 64;
    static __device__ __forceinline__ vec make(const uint4 *boards, int game, int piece)
    {
        const uint32_t k = (uint32_t)piece >> 2;
        const uint32_t word = reinterpret_cast<const uint32_t *>(boards + game)[piece & 3];
        const uint32_t eq = (((word ^ (k * 0x01010101u)) + kLo7) & kHi) ^ kHi;  // 0x80 where cell == k
        float4 v;
        v.x = __uint_as_float(prmt_sign(eq, 0u, 0x8888) & 0x3f800000u);
        v.y = __uint_as_float(prmt_sign(eq, 0u, 0x9999) & 0x3f800000u);
        v.z = __uint_as_float(prmt_sign(eq, 0u, 0xaaaa) & 0x3f800000u);
        v.w = __uint_as_float(prmt_sign(eq, 0u, 0xbbbb) & 0x3f800000u);
        return v;
    }
};

template <>
struct OneHotPiece<ML2048_ONEHOT_BF16> {  // 8 cells -> 8 bf16 = 16 bytes; 32 pieces per game
    using vec = uint4;
    static constexpr int kPiecesPerGame = 32;
    static __device__ __forceinline__ uint32_t pair(uint32_t eq, uint32_t sel)
    {
        return prmt_sign(eq, 0u, sel) & 0x3f803f80u;  // two bf16 1.0 (0x3f80) where the cells matched
    }
    static __device__ __forceinline__ vec make(const uint4 *boards, int game, int piece)
    {
        const uint32_t k = (uint32_t)piece >> 1;
        const uint32_t *w = reinterpret_cast<const uint32_t *>(boards + game) + (piece & 1) * 2;
        const uint32_t kk = k * 0x01010101u;
        const uint32_t e0 = (((w[0] ^ kk) + kLo7) & kHi) ^ kHi;
        const uint32_t e1 = (((w[1] ^ kk) + kLo7) & kHi) ^ kHi;
        return make_uint4(pair(e0, 0x9988), pair(e0, 0xbbaa), pair(e1, 0x9988), pair(e1, 0xbbaa));
    }
};

template <>
struct OneHotPiece<ML2048_ONEHOT_U8> {  // 16 cells -> 16 bytes; 16 pieces per game
    using vec = uint4;
    static constexpr int kPiecesPerGame = 16;
    static __device__ __forceinline__ vec make(const uint4 *boards, int game, int piece)
    {
        const uint4 b = boards[game];
        const uint32_t kk = (uint32_t)piece * 0x01010101u;
        return make_uint4(((((b.x ^ kk) + kLo7) & kHi) ^ kHi) >> 7, ((((b.y ^ kk) + kLo7) & kHi) ^ kHi) >> 7,
                          ((((b.z ^ kk) + kLo7) & kHi) ^ kHi) >> 7, ((((b.w ^ kk) + kLo7) & kHi) ^ kHi) >> 7);
    }
};

// Emit the one-hot rows of `games` consecutive games whose boards are in shared memory.
template <int kDtype, int kThreads>
__device__ __forceinline__ void write_onehot_tile(const uint4 *sboards, int games, void *out_base, int64_t first_game)
{
    using P = OneHotPiece<kDtype>;
    constexpr int kPer = P::kPiecesPerGame;
    static_assert(kThreads % kPer == 0, "block size must be a multiple of the pieces per game");
    constexpr int kGamesPerPass = kThreads / kPer;
    typename P::vec *out = reinterpret_cast<typename P::vec *>(out_base) + first_game * kPer;
    const int piece = threadIdx.x % kPer;
    const int g0 = threadIdx.x / kPer;
#pragma unroll 4
    for (int g = g0; g < games; g += kGamesPerPass)
        store_streaming(out + (int64_t)g * kPer + piece, P::make(sboards, g, piece));
}

// The same tile written through the TMA bulk-copy engine (large batches, 768-thread blocks): the block assembles 48 KiB of
// one-hot rows at a time in shared memory and one elected thread hands the chunk to `cp.async.bulk.global.shared::cta`
// (SASS: UBLKCP.G.S), double-buffered, so the SM issues shared-memory stores instead of global ones and the copy engine
// streams the tile to L2/HBM.  Measured at M = 2^24 against the plain-store writer above: fp32 2724 vs 2854 us per launch
// (6.67 TB/s, 102 % of the device-copy figure), bf16 1465 vs 1490 us, u8 813 vs 820 us; 24 KiB and 64 KiB chunks and
// 512/1024-thread blocks were slower.  -DML2048_ONEHOT_PLAIN switches back to plain stores.
#if !defined(ML2048_ONEHOT_PLAIN)
#define ML2048_ONEHOT_TMA 1
#endif
#if defined(ML2048_ONEHOT_TMA)
#ifndef ML2048_TMA_CHUNK_BYTES
#define ML2048_TMA_CHUNK_BYTES 49152
#endif
constexpr int kTmaChunkBytes = ML2048_TMA_CHUNK_BYTES;  // per bulk copy
#ifndef ML2048_TMA_STAGES
#define ML2048_TMA_STAGES 2
#endif
constexpr int kTmaStages = ML2048_TMA_STAGES;           // chunks staged per block

template <int kDtype, int kThreads>
__device__ __forceinline__ void write_onehot_tile_tma(const uint4 *sboards, int games, void *out_base, int64_t first_game,
                                                      uint4 *stage /* [kTmaStages][kTmaChunkBytes / 16] */)
{
    using P = OneHotPiece<kDtype>;
    constexpr int kPer = P::kPiecesPerGame;
    constexpr int kTmaChunkGames = kTmaChunkBytes / (kPer * 16);
    char *out = reinterpret_cast<char *>(out_base) + first_game * kPer * 16;
    int buf = 0;
    for (int g0 = 0; g0 < games; g0 += kTmaChunkGames, buf = (buf + 1 == kTmaStages) ? 0 : buf + 1) {
        const int n = min(kTmaChunkGames, games - g0);
        uint4 *dst = stage + buf * (kTmaChunkGames * kPer);
        // the bulk copy that last read this buffer (two chunks ago) must have finished reading it
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kTmaStages - 1) : "memory");
        __syncthreads();
        for (int q = threadIdx.x; q < n * kPer; q += kThreads) {
            const typename P::vec v = P::make(sboards, g0 + q / kPer, q % kPer);
            dst[q] = *reinterpret_cast<const uint4 *>(&v);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the async proxy
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t src = (uint32_t)__cvta_generic_to_shared(dst);
            const uint32_t bytes = (uint32_t)(n * kPer * 16);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out + (int64_t)g0 * kPer * 16), "r"(src),
                         "r"(bytes)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // smem must outlive the reads
    __syncthreads();
}
#endif

// One game's one-hot row written by a whole warp (reset path): lane l stores pieces l, l+32, ... so that one warp
// instruction covers up to 512 contiguous bytes.
template <int kDtype>
__device__ __forceinline__ void write_onehot_warp(uint4 board, void *out_base, int64_t game, int lane)
{
    using P = OneHotPiece<kDtype>;
    typename P::vec *out = reinterpret_cast<typename P::vec *>(out_base) + game * P::kPiecesPerGame;
#pragma unroll
    for (int piece = lane; piece < P::kPiecesPerGame; piece += 32)
        store_streaming(out + piece, P::make(&board, 0, piece));
}

// Calls f(std::integral_constant<int, dtype>()) for the one-hot dtype of a prepare(): the writers of the reset rows are
// compiled per dtype.  Any other value writes nothing (the host rejects it before the launch).
template <class F>
__device__ __forceinline__ void with_onehot_dtype(int dtype, F &&f)
{
    if (dtype == ML2048_ONEHOT_F32) f(std::integral_constant<int, ML2048_ONEHOT_F32>());
    else if (dtype == ML2048_ONEHOT_BF16) f(std::integral_constant<int, ML2048_ONEHOT_BF16>());
    else if (dtype == ML2048_ONEHOT_U8) f(std::integral_constant<int, ML2048_ONEHOT_U8>());
}

// The random inputs of one prepare(): scalar arguments, or the pre-drawn schedule entry a CUDA graph replays.
struct PrepDraws {
    int64_t rand_base;
    uint32_t two_mask;
    uint64_t philox_counter;
    const uint8_t *perm_table;
};

// The draws of a prepare(): the scalar arguments of `a`, or when `scheduled` the prepare() half of its schedule entry
// (prepare() draws with the entry's Philox counter, the step with the next one: step_draws).  `a` is an ml2048_prepare_args,
// or the ml2048_step_args of a step with the auto-reset fused in (reset_draws).
template <class Args>
__device__ __forceinline__ PrepDraws prep_draws(const Args &a, uint64_t philox_counter, bool scheduled)
{
    PrepDraws d{a.rand_base, a.two_mask, philox_counter, a.randperm};
    if (scheduled) {
        const ml2048_sched_entry e = a.sched[*a.sched_cursor];
        d.rand_base = e.rand_base;
        d.two_mask = e.two_mask;
        d.philox_counter = e.philox_counter;
        d.perm_table += (int64_t)e.table * a.table_stride;
    }
    return d;
}

// all 1024 boards a reset can produce and their valid-action words (board_ops.cuh): 20 KiB, L1/L2-resident
__device__ const FreshTable d_fresh = make_fresh_table();

// The two tiles a reset spawns on the empty board (game_numba.py:648-655 with :207): replay mode takes the first two
// entries of the slot's table row, Philox mode two distinct uniform cells; 2 or 4 by the table epoch's per-cell mask.
// Returns the board and (in `mask`) its valid-action word.  kLookup: both come from the 1024-entry table (the fused
// auto-reset inside the step kernel, where the reset path's LENGTH is what costs); otherwise they are computed (the
// stand-alone prepare kernels: a single latency-bound block at the training shape, where two more dependent loads from a
// cold 20 KiB table cost 0.3 us per step).
template <int kRng, bool kLookup>
__device__ __forceinline__ uint4 fresh_board(const PrepDraws &d, uint64_t slot, uint64_t philox_seed, uint32_t &mask)
{
    uint32_t c0, c1;
    if (kRng == ML2048_RNG_REPLAY) {
        const uint32_t row = ((uint32_t)d.rand_base + (uint32_t)slot) & (uint32_t)(kRandRows - 1);  // (rand_base + slot) mod 1024, both >= 0
        const uint32_t p = __ldg(reinterpret_cast<const uint32_t *>(d.perm_table) + row * 4);
        c0 = p & 15u;
        c1 = (p >> 8) & 15u;
    } else {
        const u32x2 rnd = slot_draws(slot, d.philox_counter, philox_seed, kResetStream);
        c0 = rnd.x >> 28;
        c1 = umulhi32(rnd.y, 15u);
        c1 += (c1 >= c0) ? 1u : 0u;
    }
    const uint32_t t0 = (d.two_mask >> c0) & 1u, t1 = (d.two_mask >> c1) & 1u;  // 1: the tile is a 2, 0: a 4 (game_numba.py:207)
    if (kLookup) {
        const uint32_t idx = (c0 << 6) | (c1 << 2) | (t0 << 1) | t1;
        mask = __ldg(d_fresh.mask + idx);
        return __ldg(reinterpret_cast<const uint4 *>(d_fresh.board) + idx);
    }
    uint32_t r0 = 0u, r1 = 0u, r2 = 0u, r3 = 0u;
    put_cell_shift(r0, r1, r2, r3, c0, 2u - t0);
    put_cell_shift(r0, r1, r2, r3, c1, 2u - t1);
    mask = valid_mask(r0, r1, r2, r3);
    return make_uint4(r0, r1, r2, r3);
}

// ---- what the two step kernels share --------------------------------------------------------

// What a step launch draws once: the step's random schedule.
struct StepDraws {
    int64_t rand_seed;
    uint32_t two_mask;
    uint64_t philox_counter;
    const uint8_t *keys_table;
};

// The scalar arguments, or (`scheduled`) the step half of the pre-drawn entry a CUDA graph replays, whose cursor the launch
// then advances.
__device__ __forceinline__ StepDraws step_draws(const ml2048_step_args &a, bool scheduled)
{
    StepDraws d{a.rand_seed, a.two_mask, a.philox_counter, a.randperm_keys};
    if (scheduled) {
        const int64_t cursor = *a.sched_cursor;
        const ml2048_sched_entry e = a.sched[cursor];
        d.rand_seed = e.rand_seed;
        d.two_mask = e.two_mask;
        d.philox_counter = e.philox_counter + 1ull;
        d.keys_table += (int64_t)e.table * a.table_stride;
        if (a.sched_cursor_next && blockIdx.x == 0 && threadIdx.x == 0) *a.sched_cursor_next = cursor + 1;
    }
    return d;
}

// The draws of the prepare() that a step with the auto-reset fused in stands in for.  Its 2-vs-4 mask is the step's (one
// schedule entry serves both): reusing the step's register instead of loading the entry's field again keeps the pair kernel
// from spilling more.
__device__ __forceinline__ PrepDraws reset_draws(const ml2048_step_args &a, const StepDraws &step, bool scheduled)
{
    PrepDraws d = prep_draws(a, a.prepare_philox_counter, scheduled);
    d.two_mask = step.two_mask;
    return d;
}

// Row (rand_seed + global slot) mod 1024 of the spawn keys (game_numba.py:681, :733); the low bits of the 32-bit sum are those of
// the 64-bit one.
__device__ __forceinline__ uint32_t spawn_row(int64_t rand_seed, uint64_t slot)
{
    return ((uint32_t)rand_seed + (uint32_t)slot) & (uint32_t)(kRandRows - 1);
}

// The fused auto-reset of finished game g + j (see ml2048_step_args::reset_rank): a fresh board and its mask, written back
// into the INPUT buffers (prev_state / prev_valid_actions of this step are the post-reset board and mask,
// game_numba.py:672-673), id = id_base + order (`order`: the slot-ordered rank of the game among this launch's resets,
// :641-644), entry `order` of the index list, age 0.  The caller plays the returned board from step 0, score 0; the step's own
// stores write the rest.  (The pair kernel passes its first game as a 32-bit g and j = 0 or 1, so that the reset computes its
// addresses the way the rest of that kernel does; a 64-bit g0 + j changes the SASS of the whole kernel.)
template <int kRng, typename Index>
__device__ __forceinline__ uint4 reset_in_step(const ml2048_step_args &a, const PrepDraws &d, Index g, int j, int32_t id_base,
                                               int32_t order, bool write_index, bool clear_age, uint32_t &mask)
{
    const uint4 bd = fresh_board<kRng, true>(d, (uint64_t)(a.slot_base + g + j), a.philox_seed, mask);
    reinterpret_cast<uint4 *>(const_cast<void *>(a.board_in))[g + j] = bd;
    reinterpret_cast<uint32_t *>(const_cast<void *>(a.valid_in))[g + j] = mask;
    a.id[g + j] = id_base + order;
    if (write_index && (int64_t)order < a.num_games) a.reset_indices[order] = (int64_t)g + j;
    if (clear_age) a.age[g + j] = 0;
    return bd;
}

// reward_fn (game_numba.py:728, :408-504) of a move from `old` to `now` that fused `f` and gained `gain`; kNormalReward:
// reward_fn_normal, known at compile time.
template <bool kNormalReward>
__device__ __forceinline__ float step_reward(int32_t kind, const Fusions &f, uint4 now, uint4 old, float gain)
{
    if (kNormalReward || kind == ML2048_REWARD_NORMAL) return gain;
    if (kind == ML2048_REWARD_IMPROVED) {
        // potential shaping on cell 0, game_numba.py:455-466 (all terms are exact integers in f32: |extra| <= 2^23)
        const uint32_t s0 = now.x & 0xffu, p0 = old.x & 0xffu;
        const int extra = (s0 ? (64 << s0) : 0) - (p0 ? (64 << p0) : 0);
        return gain + (float)extra;
    }
    if (kind == ML2048_REWARD_RANK) return (float)fusion_rank(f);
    if (kind == ML2048_REWARD_MAXCELL) {
        const uint32_t cur = max_cell(now.x, now.y, now.z, now.w), prev = max_cell(old.x, old.y, old.z, old.w);
        return (float)fusion_count(f) + ((cur > prev) ? (float)(1u << cur) : 0.0f);
    }
    return gain;
}

// ---- the step kernel ------------------------------------------------------------------------

// direction -> permute selectors of the move (board_ops.cuh): 128 bytes that live in L1; a game's row is fetched with two
// read-only vector loads (no shared-memory copy, so no barrier at the start of the block)
__device__ const uint32_t d_move_sel[4 * kMoveSelRow] = ML2048_MOVE_SEL_TABLE;
// ... and the same rows indexed by (valid-direction mask, k) for the in-kernel random policy (2 KiB, L1-resident)
__device__ const PolicySelTable d_policy_sel = make_policy_sel_table();

__device__ __forceinline__ uint32_t load_action(const void *actions, int dtype, int64_t g)
{
    if (dtype == ML2048_ACT_U8) return reinterpret_cast<const uint8_t *>(actions)[g];
    if (dtype == ML2048_ACT_I64) {
        const unsigned long long a = reinterpret_cast<const unsigned long long *>(actions)[g];
        return a > 3ull ? 4u : (uint32_t)a;  // negative values are huge as unsigned: invalid, like any value above 3
    }
    return (uint32_t) reinterpret_cast<const int32_t *>(actions)[g];
}

// Replaces _vec_step (game_numba.py:701-738) + the prev copies of VecGame.step (:672-673).
// kFull adds the rollout extras (policy-logits sampling, transition record, episode log); the lean variant
// compiles them out so the plain step pays nothing for them.
// kReset fuses the auto-reset (ml2048_prepare) into the step: see ml2048_step_args::reset_rank.
template <int kRng, bool kLog, int kOneHot, bool kFull, int kThreads, bool kReset = false>
// lean variants in small blocks: all 2048 thread slots of an SM filled, i.e. <= 32 registers; the variants with the rollout
// extras hold more live values and are left to the register allocator (no spills)
// (the fused-reset variants WITH a one-hot are HBM-bound and carry a few more live values: 1536 threads per SM, 42 registers)
__global__ void __launch_bounds__(kThreads, kThreads == kOneHotStepThreads              ? kOneHotStepMinBlocks
                                            : kFull                                     ? 1
                                            : (kReset && kOneHot != ML2048_ONEHOT_NONE) ? (1536 / kThreads > 32 ? 32 : 1536 / kThreads)
                                                                                        : (2048 / kThreads > 32 ? 32 : 2048 / kThreads))
    step_kernel(const ml2048_step_args a)
{
    __shared__ uint4 sboards[kOneHot != ML2048_ONEHOT_NONE ? kThreads : 1];
#if defined(ML2048_ONEHOT_TMA)
    extern __shared__ __align__(128) uint4 tma_stage[];  // [kTmaStages][kTmaChunkBytes] when launched with dynamic shared memory
#endif
    const int64_t block_first = (int64_t)blockIdx.x * kThreads;
    const int64_t g = block_first + threadIdx.x;
    const bool live = g < a.num_games;
    uint4 out_board = make_uint4(0, 0, 0, 0);

    const StepDraws draws = step_draws(a, a.sched != nullptr);

    // fused auto-reset: which lanes of this warp hold a finished game (all non-exited lanes vote; a finished game is one
    // whose mask is all zero, game_numba.py:734-735)
    uint4 bd = make_uint4(0, 0, 0, 0);
    uint32_t mask_now = 0u;   // the CURRENT valid-action word, when the variant needs it before the move
    const bool want_mask = kReset || a.action_mode != ML2048_ACTIONS_GIVEN;
    if (live) {
        bd = reinterpret_cast<const uint4 *>(a.board_in)[g];
        // The current mask is a function of the current board.  The variants with a fused one-hot are HBM-bound with
        // idle issue slots, and every extra READ stream costs a write-dominated kernel far more than its bytes (DRAM bus
        // turnarounds: tools/write_patterns.cu), so they recompute the mask (~45 instructions) instead of loading it; the
        // issue-bound core-only kernel loads it.
        if (want_mask) {
#if !defined(ML2048_LOAD_MASK)
            if (kOneHot != ML2048_ONEHOT_NONE) mask_now = valid_mask(bd.x, bd.y, bd.z, bd.w);
            else
#endif
                mask_now = reinterpret_cast<const uint32_t *>(a.valid_in)[g];
        }
    }
    bool was_reset = false;
    if (kReset) {
        asm volatile("griddepcontrol.wait;" ::: "memory");  // a programmatic dependent of the scan: see autoreset_scan_kernel
        const bool over = live && mask_now == 0u;
        const uint32_t over_lanes = __ballot_sync(0xffffffffu, over);
        if (over) {
            // rank of this slot among all finished slots (slot order): lower chunks + lower groups of the chunk + lower lanes
            // (a shard holds fewer than 2^31 games: 32-bit indices)
            const uint32_t group = (uint32_t)g >> 5;
            const int32_t order = __ldg(a.reset_chunk_base + (group >> 10)) + __ldg(a.reset_rank + group) +
                                  __popc(over_lanes & ((1u << (threadIdx.x & 31)) - 1u));
            bd = reset_in_step<kRng>(a, reset_draws(a, draws, a.sched != nullptr), g, 0, (int32_t)*a.reset_id_base, order,
                                     a.reset_indices != nullptr, a.age != nullptr, mask_now);
            was_reset = true;
        }
    }

    if (live) {
        const uint64_t slot = (uint64_t)(a.slot_base + g);
        // one uniform word per game-step from the policy stream and (Philox mode) one from the spawn stream; a Philox2x32-10
        // block serves the two slots of a pair (board_ops.cuh: slot_word)
        u32x2 rnd = {0u, 0u};  // .x picks the spawn cell (Philox mode), .y is the policy's uniform word
        if (kRng == ML2048_RNG_PHILOX) rnd.x = slot_word(slot, draws.philox_counter, a.philox_seed, kSpawnStream);
        if (a.action_mode != ML2048_ACTIONS_GIVEN) rnd.y = slot_word(slot, draws.philox_counter, a.philox_seed, 0u);
        uint32_t action;
        const auto current_mask = [&]() -> uint32_t { return mask_now; };
        const uint32_t *sel_row;  // the move's permute selectors (board_ops.cuh)
        if (a.action_mode == ML2048_ACTIONS_RANDOM_VALID) {
            // uniform over the valid directions (policy/random.py:17-27), direction 0 when the game is over: k = floor(u * nvalid)
            // indexes the (mask, k) table, whose row carries the selectors AND the direction -- no search for the k-th set bit
            const uint32_t bits = mask_bits4(current_mask());
            const uint32_t kth = umulhi32(rnd.y, popc32(bits));
            if (kThreads == kSmallStepThreads) {
                // small batches are latency-bound: the 2 KiB table costs a few more cold L1 lines per block than it saves in
                // issue slots (8.2 vs 8.5 us per step at M = 2048 in a CUDA graph), so they search the k-th set bit
                action = bits ? kth_valid_action(bits, kth) : 0u;
                sel_row = d_move_sel + action * kMoveSelRow;
            } else {
                sel_row = d_policy_sel.w + (bits * 4u + kth) * kMoveSelRow;
                action = 0u;  // read from the row below
            }
        } else if (kFull && a.action_mode == ML2048_ACTIONS_FROM_LOGITS) {
            const uint32_t bits = mask_bits4(current_mask());
            const float4 lg = reinterpret_cast<const float4 *>(a.logits)[g];
            float lp;
            action = sample_masked_categorical(lg.x, lg.y, lg.z, lg.w, bits, rnd.y, lp);
            if (a.actions_out) reinterpret_cast<uint8_t *>(a.actions_out)[g] = (uint8_t)action;
            if (a.log_prob_out) a.log_prob_out[g] = lp;
            sel_row = d_move_sel + (action & 3u) * kMoveSelRow;
        } else {
            action = load_action(a.actions, a.action_dtype, g);
            sel_row = d_move_sel + (action & 3u) * kMoveSelRow;
        }

        uint32_t r0 = bd.x, r1 = bd.y, r2 = bd.z, r3 = bd.w;
        Fusions f;
        float tr_reward = 0.0f, tr_score = 0.0f;
        int32_t tr_step = 0;
        uint32_t tr_term = 0u, tr_mask = 0u;
        const uint32_t row_action = move_board_sel(r0, r1, r2, r3, sel_row, f);
        if (a.action_mode == ML2048_ACTIONS_RANDOM_VALID) {
            if (kThreads != kSmallStepThreads) action = row_action;
            if (a.actions_out) reinterpret_cast<uint8_t *>(a.actions_out)[g] = (uint8_t)action;
        }
        // valid_actions[action] (game_numba.py:718) == "the move changes the board"; out-of-range
        // actions (which the reference would index out of bounds with) count as invalid moves
        const bool moved = (action < 4u) && (((r0 ^ bd.x) | (r1 ^ bd.y) | (r2 ^ bd.z) | (r3 ^ bd.w)) != 0u);

        if (moved) {
            // reward_fn (:728) and the score increment (:729-731)
            const float gain = fusion_gain(f);  // an exact integer < 2^22
            const float reward = step_reward<false>(a.reward_kind, f, make_uint4(r0, r1, r2, r3), bd, gain);
            // step count and score are the halves of ONE 8-byte record per game: one load, one store, one stream
            int2 *const step_score = reinterpret_cast<int2 *>(a.step) + g;
            // a game reset by this very launch starts from step 0, score 0 (its record still holds the finished game's)
            const int2 old_ss = (kReset && was_reset) ? make_int2(0, 0) : *step_score;
            const float score = __int_as_float(old_ss.y) + gain;
            const int32_t nstep = old_ss.x + 1;

            // spawn one tile (_spawn2 with count = 1, game_numba.py:733)
            const uint32_t n0 = occupied_signs(r0), n1 = occupied_signs(r1), n2 = occupied_signs(r2), n3 = occupied_signs(r3);
            uint32_t cell;
            if (kRng == ML2048_RNG_REPLAY) {
                const uint4 keys = __ldg(reinterpret_cast<const uint4 *>(draws.keys_table) + spawn_row(draws.rand_seed, slot));
                // a move that changed the board leaves at least one empty cell (a slide vacates one, a fusion frees
                // one), so the search cannot come back empty-handed here
                cell = first_empty_key(keys.x, keys.y, keys.z, keys.w, n0, n1, n2, n3) & 15u;
            } else {
                const uint32_t empties = empties16(~n0 & kHi, ~n1 & kHi, ~n2 & kHi, ~n3 & kHi);
                const uint32_t ne = popc32(empties);  // >= 1, see above
                cell = kth_set_bit16(empties, umulhi32(rnd.x, ne));
            }
            // 2 or 4: tied to the CELL for the table epoch in force (game_numba.py:207), in both modes
            const uint32_t value = 2u - ((draws.two_mask >> cell) & 1u);
            if (kThreads == kSmallStepThreads) put_cell_shift(r0, r1, r2, r3, cell, value);  // latency-bound: no table load
            else put_cell(r0, r1, r2, r3, cell, value);

            const uint32_t vm = valid_mask(r0, r1, r2, r3);
            const bool dead = vm == 0u;
            reinterpret_cast<uint32_t *>(a.valid_out)[g] = vm;
            a.reward[g] = reward;
            *step_score = make_int2(nstep, __float_as_int(score));
            a.terminated[g] = dead ? 1 : 0;
            a.invalid[g] = 0;
            if (kLog) {
                uint32_t m0, m1, m2, m3;
                fusion_log(f, m0, m1, m2, m3);
                reinterpret_cast<uint4 *>(a.merged)[g] = make_uint4(m0, m1, m2, m3);
            }
            tr_reward = reward, tr_score = score, tr_step = nstep, tr_term = dead ? 1 : 0, tr_mask = vm;
            if (kFull && dead && a.episode_max_tile) {
                // eval_perf.py semantics: episodes are keyed by game id, not by finishing order
                const int64_t e = (int64_t)a.id[g] - a.episode_id_base;
                if (e >= 0 && e < a.episode_capacity) {
                    a.episode_steps[e] = nstep;
                    a.episode_score[e] = score;
                    a.episode_max_tile[e] = (uint8_t)max_cell(r0, r1, r2, r3);
                }
            }
            if (dead && a.stats) {
                // finished-episode statistics (RunnerStats, runner.py:158-166): rare (~1% of moves)
                ml2048_stats *st = a.stats + (blockIdx.x % ML2048_STATS_REPLICAS);
                const unsigned long long sc = (unsigned long long)score;
                atomicAdd(&st->max_tile_hist[min(max_cell(r0, r1, r2, r3), 19u)], 1ull);
                atomicAdd(&st->episodes, 1ull);
                atomicAdd(&st->score_sum, sc);
                atomicAdd(&st->step_sum, (unsigned long long)nstep);
                atomicMax(&st->score_max, sc);
            }
        } else {
            // invalid move: only `invalid` changes (game_numba.py:737-738); the board is carried over
            r0 = bd.x, r1 = bd.y, r2 = bd.z, r3 = bd.w;
            tr_mask = valid_mask(r0, r1, r2, r3);
            reinterpret_cast<uint32_t *>(a.valid_out)[g] = tr_mask;
            a.invalid[g] = 1;
            if (kFull) {  // stale values are recorded stale (run_train3.py:146-148)
                if (a.tr_reward) tr_reward = a.reward[g];
                if (a.tr_step) tr_step = a.step[2 * g];
                if (a.tr_terminated) tr_term = a.terminated[g];
            }
        }
        out_board = make_uint4(r0, r1, r2, r3);
        reinterpret_cast<uint4 *>(a.board_out)[g] = out_board;
        if (kFull && a.traj_state) {
            // ReplayRecorder on the device (replay.py:161-201): one row per runner step of a recorded game
            const int32_t row = a.age[g];
            const bool was_over = !moved && a.terminated[g];  // finished games idle until prepare(): not recorded again
            const int64_t e = (int64_t)a.id[g] - a.traj_id_base;
            if (!was_over && e >= 0 && e < a.traj_capacity) {
                const bool dead_now = moved && tr_term;
                const float sc = moved ? tr_score : a.score[2 * g];  // after this step (stale on an invalid move, like result["score"])
                if (row < a.traj_max_rows) {
                    const int64_t k = e * a.traj_max_rows + row;
                    reinterpret_cast<uint4 *>(a.traj_state)[k] = bd;
                    a.traj_action[k] = (int8_t)action;
                    a.traj_score[k] = sc;
                }
                if (dead_now && row + 1 < a.traj_max_rows) {
                    const int64_t k = e * a.traj_max_rows + row + 1;
                    reinterpret_cast<uint4 *>(a.traj_state)[k] = out_board;
                    a.traj_action[k] = 0;
                    a.traj_score[k] = sc;
                }
                const int64_t rows = (int64_t)row + 1 + (dead_now ? 1 : 0);
                a.traj_rows[e] = (int32_t)(rows < a.traj_max_rows ? rows : a.traj_max_rows);
            }
            if (!was_over) a.age[g] = row + 1;
        }
        if (kFull) {  // transition record (REPLAY_SPEC row, replay.py:10-20)
            if (a.tr_state) reinterpret_cast<uint4 *>(a.tr_state)[g] = bd;
            if (a.tr_valid_actions)
                reinterpret_cast<uint32_t *>(a.tr_valid_actions)[g] =
                    want_mask ? mask_now : reinterpret_cast<const uint32_t *>(a.valid_in)[g];
            if (a.tr_action) a.tr_action[g] = (int8_t)action;
            if (a.tr_reward) a.tr_reward[g] = tr_reward;
            if (a.tr_next_state) reinterpret_cast<uint4 *>(a.tr_next_state)[g] = out_board;
            if (a.tr_next_valid_actions) reinterpret_cast<uint32_t *>(a.tr_next_valid_actions)[g] = tr_mask;
            if (a.tr_step) a.tr_step[g] = tr_step;
            if (a.tr_terminated) a.tr_terminated[g] = (uint8_t)tr_term;
        }
    }

    if (kOneHot != ML2048_ONEHOT_NONE) {
        sboards[threadIdx.x] = out_board;
        __syncthreads();
        const int64_t remaining = a.num_games - block_first;
        const int games = remaining < kThreads ? (int)remaining : kThreads;
        constexpr int kOH = kOneHot == ML2048_ONEHOT_NONE ? ML2048_ONEHOT_F32 : kOneHot;
#if defined(ML2048_ONEHOT_TMA)
        if (kThreads == kOneHotStepThreads)
            write_onehot_tile_tma<kOH, kThreads>(sboards, games, a.onehot_out, block_first, tma_stage);
        else
#endif
            write_onehot_tile<kOH, kThreads>(sboards, games, a.onehot_out, block_first);
    }
}

// ---- the lean step kernel, two games per thread ---------------------------------------------
// The core-only step (no one-hot, no `merged`, none of the rollout extras) is bound by the integer ALU pipe, and a good
// part of what it issues there is not game arithmetic: two instructions of address arithmetic for each of nine arrays, the
// bounds checks, the predicates of the schedule.  A thread that owns TWO ADJACENT games computes every address once (the
// second game sits at an immediate offset), shares the prologue, and gives the scheduler two independent instruction
// streams.  Same arithmetic per game as step_kernel (the same board_ops.cuh functions in the same order, and the functions both
// kernels share: step_draws, reset_draws, reset_in_step, step_reward, spawn_row), same draws (the words of the Philox blocks of
// the global slot PAIR, which the thread computes once for both of its games), so every array is
// bit-identical to the one-game-per-thread kernel (tests/test_pair_kernel.py); large batches of the lean configuration are
// routed here by launch_step.
// Measured at M = 2^24 (auto-reset fused + random policy / given actions, us per launch):
//   before the round-2 instruction cuts (one-game-per-thread kernel: 274.6 / 231): 256 threads x 5 blocks (48 registers) 274.7 / 230.9,
//   x 4 (64) 278.2 / 240.0, x 6 (40) 270.9 / 225.2, x 8 (32, spills) 276.1 / 232.4; 128 threads x 8 (64) 270.4 / 227.9, x 10 (48)
//   273.0 / 226.8, x 12 (40 registers) 269.4 / 222.2;
//   after them (profiles/pair_kernel_variants_r02_s.txt): 128 x 12 240.7 / 196.6, 128 x 10 243.9 / 207.1, 128 x 8 247.2 / 207.5,
//   256 x 6 242.8 / 198.6, 64 x 24 241.4 / 197.4, 128 x 16 (32 registers, spills) 257.0 / 210.4.
#ifndef ML2048_PAIR_THREADS
#define ML2048_PAIR_THREADS 128
#endif
#ifndef ML2048_PAIR_MIN_BLOCKS
#define ML2048_PAIR_MIN_BLOCKS 12
#endif
constexpr int kPairThreads = ML2048_PAIR_THREADS;
constexpr int64_t kPairMinGames = 1 << 17;  // below this the batch is latency-bound: more, smaller threads win

// What launch_step works out on the host for the pair kernel and passes as a second kernel parameter: the Philox round keys of
// the two streams (functions of the seed alone; derived per warp on the uniform datapath they cost ~15 issue slots per warp)
// and one bit per optional output, so that the kernel tests a flag instead of loading and comparing a 64-bit pointer.
struct PairConst {
    PhiloxKeys policy_keys, spawn_keys;
    uint32_t flags;
};
enum : uint32_t { kPairActionsOut = 1u, kPairStats = 2u, kPairAge = 4u, kPairResetIndices = 8u, kPairOddSlotBase = 16u, kPairSched = 32u };

// What a thread reads of its two games before it can do anything: 56 bytes, three streams
struct PairLoad {
    uint4 bd[2];
    uint32_t mask[2];
    int2 ss[2];
};

// (Loading the three input streams with L1::no_allocate, to keep the lookup tables L1-resident, measured SLOWER -- 264 against
// 240 us for the fused step at M = 2^24: the two games of a pair share 32-byte sectors, and the second load of each then
// misses L1 as well.)
template <typename T>
__device__ __forceinline__ T load_stream(const T *p) { return *p; }

template <bool kWantMask>
__device__ __forceinline__ void pair_load(const ml2048_step_args &a, uint32_t g0, bool live0, bool live1, PairLoad &L)
{
    L.bd[0] = L.bd[1] = make_uint4(0, 0, 0, 0);
    L.mask[0] = L.mask[1] = 1u;
    L.ss[0] = L.ss[1] = make_int2(0, 0);
    const uint4 *board_in = reinterpret_cast<const uint4 *>(a.board_in) + g0;
    const uint32_t *valid_in = reinterpret_cast<const uint32_t *>(a.valid_in) + g0;
    const int2 *step_score = reinterpret_cast<const int2 *>(a.step) + g0;
    if (live0) {
        L.bd[0] = load_stream(board_in);
        if (kWantMask) L.mask[0] = load_stream(valid_in);
        L.ss[0] = load_stream(step_score);
    }
    if (live1) {
        L.bd[1] = load_stream(board_in + 1);
        if (kWantMask) L.mask[1] = load_stream(valid_in + 1);
        L.ss[1] = load_stream(step_score + 1);
    }
}

__device__ __forceinline__ void red_add_u64(unsigned long long *p, unsigned long long v)
{
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void red_max_u64(unsigned long long *p, unsigned long long v)
{
    asm volatile("red.global.max.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Where a game-step finds its lookup tables: the L1-resident copies in global memory.  (A policy class, so that a kernel
// with the tables elsewhere can share pair_body: see the software-pipelined experiment below.)
struct GlobalTables {
    const uint4 *keys;  // spawn keys of the table epoch in force, 1024 rows
    __device__ __forceinline__ SelRow policy_row(uint32_t index) const  // row of the (mask, k) table
    {
        const uint4 *row = reinterpret_cast<const uint4 *>(d_policy_sel.w) + index * 2u;
        const uint4 sa = __ldg(row), sb = __ldg(row + 1);
        return SelRow{sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z};
    }
    __device__ __forceinline__ SelRow move_row(uint32_t action) const
    {
        const uint4 *row = reinterpret_cast<const uint4 *>(d_move_sel) + action * 2u;
        const uint4 sa = __ldg(row), sb = __ldg(row + 1);
        return SelRow{sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z};
    }
    __device__ __forceinline__ uint4 keys_row(uint32_t row) const { return __ldg(keys + row); }
    __device__ __forceinline__ uint4 cell_entry(uint32_t cell) const { return __ldg(reinterpret_cast<const uint4 *>(d_cell_one.w) + cell); }
};

// kRandom: the in-kernel random-valid policy (else caller-given actions); kNormalReward: reward_fn_normal (else the
// reward kind is looked up at run time) -- compile-time switches for what is uniform over a launch, each worth a handful of
// issue slots per game (parameter load, compare, branch).
// All 32 lanes of a warp call this together (the fused auto-reset votes); a lane past the end of the batch has live0 = false.
template <int kRng, bool kReset, bool kRandom, bool kNormalReward, class Tables>
__device__ __forceinline__ void pair_body(const ml2048_step_args &a, const PairConst &x, const StepDraws &draws, const Tables &tab,
                                          uint32_t g0, bool live0, bool live1, PairLoad &L)
{
    // one address per array; the second game of the pair is the next element
    uint4 *board_out = reinterpret_cast<uint4 *>(a.board_out) + g0;
    uint32_t *valid_out = reinterpret_cast<uint32_t *>(a.valid_out) + g0;
    int2 *step_score = reinterpret_cast<int2 *>(a.step) + g0;
    float *reward_out = a.reward + g0;
    uint8_t *terminated = a.terminated + g0, *invalid = a.invalid + g0;

    uint4 (&bd)[2] = L.bd;
    uint32_t (&mask_now)[2] = L.mask;
    int2 (&ss)[2] = L.ss;
    const bool want_mask = kReset || kRandom;
    // With the auto-reset fused in every game moves, so the five narrow results of the pair are known together and go out as
    // ONE store per array (8 + 8 + 16 + 2 + 2 bytes) when the arrays are aligned for it: five store instructions and their
    // address arithmetic less per pair (237 against 239.5 us at M = 2^24).  Not in Philox mode, whose extra live values then spill
    // (252 against 245 us), and not for the variants without the fused reset, where holding the first game's results until the
    // second one is known to have moved costs more than the stores (given actions 213 against 198 us).
    constexpr bool kPairStores = kReset && kRng == ML2048_RNG_REPLAY;
    const bool pair_stores = kPairStores && live1 &&
                             ((reinterpret_cast<uintptr_t>(a.valid_out) | reinterpret_cast<uintptr_t>(a.reward)) & 7u) == 0u &&
                             (reinterpret_cast<uintptr_t>(a.step) & 15u) == 0u &&
                             ((reinterpret_cast<uintptr_t>(a.terminated) | reinterpret_cast<uintptr_t>(a.invalid)) & 1u) == 0u;
    uint32_t pair_vm[2] = {0u, 0u}, pair_dead[2] = {0u, 0u};
    float pair_reward[2] = {0.0f, 0.0f};
    int2 pair_ss[2] = {make_int2(0, 0), make_int2(0, 0)};

    if (kReset) {
        // (launched as a programmatic dependent of the scan: everything above overlapped it; from here on the kernel reads the
        // scan's results and writes the `terminated` flags the scan reads.  A no-op when not launched that way.)
        asm volatile("griddepcontrol.wait;" ::: "memory");
        // fused auto-reset (reset_in_step): lane l holds slots 2l and 2l+1 of the warp's 64, i.e. of TWO 32-slot groups
        // of the scan; ranks count the finished games of the lower lanes of the same half-warp, both games of each
        const bool over0 = live0 && mask_now[0] == 0u, over1 = live1 && mask_now[1] == 0u;
        const uint32_t lanes0 = __ballot_sync(0xffffffffu, over0), lanes1 = __ballot_sync(0xffffffffu, over1);
        if (over0 || over1) {
            const uint32_t lane = threadIdx.x & 31u;
            const uint32_t lower = ((1u << lane) - 1u) & (0xffffu << (lane & 16u));
            // (asking for the two rank words up front, together with the boards, so that the reset path has one dependent round
            // trip less, measured no different: 239.5 against 239.6 us -- the kernel is not latency-bound)
            const uint32_t group = g0 >> 5;
            int32_t order = __ldg(a.reset_chunk_base + (group >> 10)) + __ldg(a.reset_rank + group) + __popc(lanes0 & lower) +
                            __popc(lanes1 & lower);
            const PrepDraws d = reset_draws(a, draws, x.flags & kPairSched);
            const int32_t id_base = (int32_t)*a.reset_id_base;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                if (j == 0 ? over0 : over1) {
                    bd[j] = reset_in_step<kRng>(a, d, g0, j, id_base, order, x.flags & kPairResetIndices, x.flags & kPairAge, mask_now[j]);
                    ss[j] = make_int2(0, 0);
                    order += 1;
                }
            }
        }
    }
    if (!live0) return;

    // the uniform words of the two games: one Philox block per stream serves both when the thread's first global slot is
    // even (always, unless a shard starts at an odd slot)
    const uint64_t slot0 = (uint64_t)(a.slot_base + g0);
    uint32_t policy_word[2] = {0u, 0u}, spawn_word[2] = {0u, 0u};
    if (kRandom) {
        if (!(x.flags & kPairOddSlotBase)) {
            const u32x2 b = slot_draws_keys(slot0 >> 1, draws.philox_counter, x.policy_keys);
            policy_word[0] = b.x, policy_word[1] = b.y;
        } else {
            policy_word[0] = slot_word_keys(slot0, draws.philox_counter, x.policy_keys);
            policy_word[1] = slot_word_keys(slot0 + 1, draws.philox_counter, x.policy_keys);
        }
    }
    if (kRng == ML2048_RNG_PHILOX) {
        if (!(x.flags & kPairOddSlotBase)) {
            const u32x2 b = slot_draws_keys(slot0 >> 1, draws.philox_counter, x.spawn_keys);
            spawn_word[0] = b.x, spawn_word[1] = b.y;
        } else {
            spawn_word[0] = slot_word_keys(slot0, draws.philox_counter, x.spawn_keys);
            spawn_word[1] = slot_word_keys(slot0 + 1, draws.philox_counter, x.spawn_keys);
        }
    }

#pragma unroll
    for (int j = 0; j < 2; ++j) {
        if (j == 1 && !live1) break;
        const uint32_t g = g0 + j;
        const uint64_t slot = slot0 + j;
        const u32x2 rnd = {spawn_word[j], policy_word[j]};
        uint32_t action = 0u;
        SelRow sel_row;
        if (kRandom) {
            const uint32_t bits = mask_bits4(mask_now[j]);
            sel_row = tab.policy_row(bits * 4u + umulhi32(rnd.y, popc32(bits)));
        } else {
            action = load_action(a.actions, a.action_dtype, g);
            sel_row = tab.move_row(action & 3u);
        }
        uint32_t r0 = bd[j].x, r1 = bd[j].y, r2 = bd[j].z, r3 = bd[j].w;
        Fusions f;
        const uint32_t row_action = move_board_row(r0, r1, r2, r3, sel_row, f);
        if (kRandom) {
            action = row_action;
            if (x.flags & kPairActionsOut) reinterpret_cast<uint8_t *>(a.actions_out)[g] = (uint8_t)action;
        }
        // valid_actions[action] (game_numba.py:718) == "the move changes the board".  The random policy only ever picks a valid
        // direction, so there the move counts exactly when the game has one (mask != 0): no comparison of the boards.  And with
        // the auto-reset fused in, every game has one: a finished game was just replaced by a fresh board (two tiles: never stuck)
        const bool moved = kReset   ? true
                           : kRandom ? mask_now[j] != 0u
                                     : (action < 4u) && (((r0 ^ bd[j].x) | (r1 ^ bd[j].y) | (r2 ^ bd[j].z) | (r3 ^ bd[j].w)) != 0u);
        if (moved) {
            const float gain = fusion_gain(f);
            const float reward = step_reward<kNormalReward>(a.reward_kind, f, make_uint4(r0, r1, r2, r3), bd[j], gain);
            const float score = __int_as_float(ss[j].y) + gain;
            const int32_t nstep = ss[j].x + 1;
            const uint32_t n0 = occupied_signs(r0), n1 = occupied_signs(r1), n2 = occupied_signs(r2), n3 = occupied_signs(r3);
            uint32_t cell;
            if (kRng == ML2048_RNG_REPLAY) {
                const uint4 keys = tab.keys_row(spawn_row(draws.rand_seed, slot));
                cell = first_empty_key(keys.x, keys.y, keys.z, keys.w, n0, n1, n2, n3) & 15u;
            } else {
                const uint32_t empties = empties16(~n0 & kHi, ~n1 & kHi, ~n2 & kHi, ~n3 & kHi);
                cell = kth_set_bit16(empties, umulhi32(rnd.x, popc32(empties)));
            }
            put_cell_entry(r0, r1, r2, r3, tab.cell_entry(cell), 2u - ((draws.two_mask >> cell) & 1u));
            const uint32_t vm = valid_mask(r0, r1, r2, r3);
            const bool dead = vm == 0u;
            if (kPairStores && pair_stores) {
                pair_vm[j] = vm, pair_reward[j] = reward, pair_ss[j] = make_int2(nstep, __float_as_int(score)), pair_dead[j] = dead ? 1u : 0u;
            } else {
                valid_out[j] = vm;
                reward_out[j] = reward;
                step_score[j] = make_int2(nstep, __float_as_int(score));
                terminated[j] = dead ? 1 : 0;
                invalid[j] = 0;
            }
            if (dead && (x.flags & kPairStats)) {
                // (plain reductions: a warp has one or two finished games, so the vote / elect code the compiler wraps around
                // atomicAdd to aggregate a warp's contributions costs more instructions than it saves transactions)
                ml2048_stats *st = a.stats + (blockIdx.x % ML2048_STATS_REPLICAS);
                const unsigned long long sc = (unsigned long long)score;
                red_add_u64(&st->max_tile_hist[min(max_cell(r0, r1, r2, r3), 19u)], 1ull);
                red_add_u64(&st->episodes, 1ull);
                red_add_u64(&st->score_sum, sc);
                red_add_u64(&st->step_sum, (unsigned long long)nstep);
                red_max_u64(&st->score_max, sc);
            }
        } else {
            r0 = bd[j].x, r1 = bd[j].y, r2 = bd[j].z, r3 = bd[j].w;
            valid_out[j] = want_mask ? mask_now[j] : valid_mask(r0, r1, r2, r3);
            invalid[j] = 1;
        }
        board_out[j] = make_uint4(r0, r1, r2, r3);
    }
    if (kPairStores && pair_stores) {
        *reinterpret_cast<uint2 *>(valid_out) = make_uint2(pair_vm[0], pair_vm[1]);
        *reinterpret_cast<float2 *>(reward_out) = make_float2(pair_reward[0], pair_reward[1]);
        *reinterpret_cast<int4 *>(step_score) = make_int4(pair_ss[0].x, pair_ss[0].y, pair_ss[1].x, pair_ss[1].y);
        *reinterpret_cast<uint16_t *>(terminated) = (uint16_t)(pair_dead[0] | (pair_dead[1] << 8));
        *reinterpret_cast<uint16_t *>(invalid) = 0;
    }
}

// one pair per thread
template <int kRng, bool kReset, bool kRandom, bool kNormalReward>
__global__ void __launch_bounds__(kPairThreads, ML2048_PAIR_MIN_BLOCKS) step_pair_kernel(const ml2048_step_args a, const PairConst x)
{
    const uint32_t n = (uint32_t)a.num_games;  // < 2^31: launch_step
    const uint32_t warp_first = (blockIdx.x * kPairThreads + (threadIdx.x & ~31u)) * 2u;
    if (warp_first >= n) return;
    const uint32_t g0 = (blockIdx.x * kPairThreads + threadIdx.x) * 2u;  // this thread owns games g0 and g0 + 1
    const bool live0 = g0 < n, live1 = g0 + 1u < n;
    // the 56 input bytes are requested before anything else is looked at: every instruction ahead of these loads is DRAM
    // latency the warp cannot hide behind its own work
    PairLoad L;
    pair_load<kReset || kRandom>(a, g0, live0, live1, L);
    const StepDraws draws = step_draws(a, x.flags & kPairSched);
    const GlobalTables tab{reinterpret_cast<const uint4 *>(draws.keys_table)};
    pair_body<kRng, kReset, kRandom, kNormalReward>(a, x, draws, tab, g0, live0, live1, L);
}

// A software-pipelined variant of this kernel was built and measured in round 2 and is NOT kept (profiles/pair_loop_experiments_r02.txt): a
// GPU-filling grid striding over the batch, every thread prefetching the 56 input bytes of its next pair while it plays the
// current one.  (1) Prefetch into registers (56 registers, 9 blocks per SM): 293 us against 240 us for the fused step at
// M = 2^24 -- ptxas put the prefetch on a scoreboard that loads of the body share, so the first of them waits for the DRAM round
// trip anyway (ncu: 20 % of all stall samples on that one instruction).  (2) Prefetch with cp.async into shared memory (no
// destination registers, 40 registers, every thread waiting only for its own copies): 328 us -- the staging buffers leave
// little L1 and the table lookups in the middle of every dependency chain then miss it.  (3) The same with the tables in
// shared memory as well (512-thread blocks, one buffer): 324 us, issue slots 51 % busy against 66 %: with the DRAM waits gone
// the warps wait for the reset path's dependent loads, the shared-memory lookups (`short scoreboard` 2.5 warps per issue)
// and the LSU queue (`mio throttle`) instead.  (4) 128-thread blocks, twelve per SM, ONE 7 KiB cp.async buffer per block (L1
// keeps ~120 KiB for the tables, which stay in global memory), on the final kernel: 299 us against 230 us, and 288 against 198 us
// without the fused reset.  One pair per thread with twelve 128-thread blocks per SM stays the fastest: what the loop loses is not
// explained by any single stall reason -- blocks that start and finish at different times keep the demand on the ALU pipe smooth,
// blocks that march through the batch together do not.

// ---- auto-reset (VecGame.prepare, game_numba.py:619-658) -----------------------------------
// Pass 1: terminated games per tile of 4096 slots.  Pass 2: exclusive scan over tiles (one block),
// advances the id counter.  Pass 3: per tile, slot-ordered offsets -> ids, reset indices, fresh boards.

__device__ __forceinline__ uint32_t flags16(uint4 t)  // sixteen 0/1 bytes -> 16-bit mask
{
    const uint32_t m = 0x10204080u;  // gathers bits 0,8,16,24 into the top nibble
    return ((t.x * m) >> 28) | (((t.y * m) >> 24) & 0xf0u) | (((t.z * m) >> 20) & 0xf00u) | (((t.w * m) >> 16) & 0xf000u);
}

// Inclusive scan of `v` over the first kWidth lanes of a warp (all 32 lanes take part).
template <int kWidth>
__device__ __forceinline__ int warp_inclusive_scan(int v)
{
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < kWidth; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += n;
    }
    return v;
}

// Block-wide exclusive scan of `v` over a block of kThreads threads (a multiple of 32): `below` = the sum over the lower
// threads, `total` = the sum over the block, both in every thread.  One barrier; `warp_tot` (kThreads / 32 ints of shared
// memory) may be written again only after another one.
struct BlockScan {
    int below, total;
};

template <int kThreads>
__device__ __forceinline__ BlockScan block_scan(int v, int *warp_tot)
{
    static_assert(kThreads % 32 == 0 && kThreads <= 1024, "a block of whole warps");
    constexpr int kWarps = kThreads / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int inc = warp_inclusive_scan<32>(v);
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    // every warp scans the warp totals itself: no second barrier
    const int t = lane < kWarps ? warp_tot[lane] : 0;
    const int w = warp_inclusive_scan<kWarps>(t);
    return BlockScan{__shfl_sync(0xffffffffu, w - t, warp) + inc - v, __shfl_sync(0xffffffffu, w, kWarps - 1)};
}

// Exclusive scan of in[0, n) into out[0, n) (`in` may be `out`) by one block of kThreads threads (the block size it is
// launched with), in passes of kThreads entries that carry the running total from one to the next.  Returns the grand total to
// every thread.
template <int kThreads>
__device__ __forceinline__ int block_scan_passes(const volatile int32_t *in, int32_t *out, int n, int *warp_tot)
{
    int carry = 0;
    for (int base = 0; base < n; base += kThreads) {
        const int i = base + threadIdx.x;
        const BlockScan s = block_scan<kThreads>(i < n ? in[i] : 0, warp_tot);
        if (i < n) out[i] = carry + s.below;
        carry += s.total;
        __syncthreads();  // warp_tot is written again by the next pass
    }
    return carry;
}

__global__ void __launch_bounds__(kPrepThreads) prepare_count_kernel(const uint4 *term16, int64_t n16, int32_t *tile_counts)
{
    __shared__ int warp_tot[kPrepThreads / 32];
    const int64_t i = (int64_t)blockIdx.x * kPrepThreads + threadIdx.x;
    int c = 0;
    if (i < n16) c = __popc(flags16(term16[i]));
    const int total = block_scan<kPrepThreads>(c, warp_tot).total;
    if (threadIdx.x == 0) tile_counts[blockIdx.x] = total;
}

constexpr int kPrepScanThreads = 1024;  // the single block of prepare_scan_kernel

// scratch layout: [0, tiles) tile counts -> exclusive offsets; then (8-byte aligned) int64 id_base
__global__ void __launch_bounds__(kPrepScanThreads) prepare_scan_kernel(int32_t *tile_counts, int tiles, int64_t *id_base_slot,
                                                                        int64_t *game_count, int advance, int64_t *reset_count)
{
    __shared__ int warp_tot[kPrepScanThreads / 32];
    const int total = block_scan_passes<kPrepScanThreads>(tile_counts, tile_counts, tiles, warp_tot);
    if (threadIdx.x == 0) {
        const int64_t base = *game_count;
        *id_base_slot = base;
        if (advance) *game_count = base + total;
        *reset_count = total;
    }
}

// The reset body of VecGame.prepare for ONE slot (game_numba.py:634-656): zero the record, id = id_base + order (the
// rank of the slot among all slots reset by this call: slot-ordered like :641-644), two spawned tiles, the mask.
// Returns the fresh board.
template <int kRng>
__device__ __forceinline__ uint4 reset_slot(const ml2048_prepare_args &a, const PrepDraws &d, int64_t g, int64_t order, int64_t id_base)
{
    uint32_t fresh_mask;
    const uint4 bd = fresh_board<kRng, false>(d, (uint64_t)(a.slot_base + g), a.philox_seed, fresh_mask);
    reinterpret_cast<uint4 *>(a.board)[g] = bd;
    reinterpret_cast<uint32_t *>(a.valid)[g] = fresh_mask;
    a.id[g] = (int32_t)(id_base + order);
    reinterpret_cast<int2 *>(a.step)[g] = make_int2(0, 0);  // step = 0, score = 0.0f: one store
    a.reward[g] = 0.0f;
    a.invalid[g] = 0;
    if (a.merged) reinterpret_cast<uint4 *>(a.merged)[g] = make_uint4(0, 0, 0, 0);
    if (a.age) a.age[g] = 0;
    if (a.reset_indices) a.reset_indices[order] = g;
    return bd;
}

// The one-hot rows of the games the lanes of a warp just reset (`has`), written by the whole warp one game after the
// other so that every store instruction covers 512 contiguous bytes.
__device__ __forceinline__ void write_onehot_of_lanes(const ml2048_prepare_args &a, bool has, uint4 bd, long long g, int lane)
{
    uint32_t ballot = __ballot_sync(0xffffffffu, has);
    while (ballot) {
        const int src = __ffs((int)ballot) - 1;
        ballot &= ballot - 1u;
        const uint4 b = make_uint4(__shfl_sync(0xffffffffu, bd.x, src), __shfl_sync(0xffffffffu, bd.y, src),
                                   __shfl_sync(0xffffffffu, bd.z, src), __shfl_sync(0xffffffffu, bd.w, src));
        const long long gg = __shfl_sync(0xffffffffu, g, src);
        with_onehot_dtype(a.onehot_dtype, [&](auto k) { write_onehot_warp<decltype(k)::value>(b, a.onehot, gg, lane); });
    }
}

// Reset pass over one tile of 4096 slots by one block.  `tile_offset` = finished games in earlier tiles, `id_base` = id of
// the first game reset by this prepare().  Returns the number of games this tile reset (to every thread).
template <int kRng>
__device__ __forceinline__ int apply_tile(const ml2048_prepare_args &a, int64_t tile, int64_t tile_offset, int64_t id_base,
                                          int *warp_tot)
{
    const int64_t n16 = (a.num_games + 15) / 16;
    const int64_t i = tile * kPrepThreads + threadIdx.x;
    uint32_t mask = 0u;
    if (i < n16) mask = flags16(reinterpret_cast<const uint4 *>(a.terminated)[i]);
    const BlockScan s = block_scan<kPrepThreads>(__popc(mask), warp_tot);
    const bool had_any = mask != 0u;
    const int lane = threadIdx.x & 31;
    const PrepDraws draws = prep_draws(a, a.philox_counter, a.sched != nullptr);
    int64_t order = tile_offset + s.below;  // rank among all reset slots

    // rounds: in each one every lane that still has a finished game resets one; the one-hot rows of the round
    // are then written by the whole warp, one game after the other
    while (__any_sync(0xffffffffu, mask != 0u)) {
        const bool has = mask != 0u;
        uint4 bd = make_uint4(0u, 0u, 0u, 0u);
        long long g = 0;
        if (has) {
            const int j = __ffs((int)mask) - 1;
            mask &= mask - 1u;
            g = i * 16 + j;
            bd = reset_slot<kRng>(a, draws, g, order, id_base);
            order += 1;
        }
        if (a.onehot) write_onehot_of_lanes(a, has, bd, g, lane);
    }
    // every flag this thread saw is now cleared (entry.fill(0), game_numba.py:638-639)
    if (had_any) reinterpret_cast<uint4 *>(a.terminated)[i] = make_uint4(0, 0, 0, 0);
    return s.total;
}

template <int kRng>
__global__ void __launch_bounds__(kPrepThreads) prepare_apply_kernel(const ml2048_prepare_args a, const int32_t *tile_offsets,
                                                                     const int64_t *id_base_slot)
{
    __shared__ int warp_tot[kPrepThreads / 32];
    const int64_t id_base = *id_base_slot + (a.id_offset ? *a.id_offset : 0);
    apply_tile<kRng>(a, blockIdx.x, tile_offsets[blockIdx.x], id_base, warp_tot);
}

// Small batches (a few tiles): count, scan and reset in ONE single-block launch -- the tiles are walked in order, so
// the running total IS the exclusive scan.  Saves two launches per prepare(), which is what a 2048-game step costs.
constexpr int kPrepSmallMaxGames = 2 * kPrepTile;  // beyond two tiles the serial walk loses to the three-kernel path

template <int kRng>
__global__ void __launch_bounds__(kPrepThreads) prepare_small_kernel(const ml2048_prepare_args a)
{
    __shared__ int warp_tot[kPrepThreads / 32];
    const int tiles = (int)((a.num_games + kPrepTile - 1) / kPrepTile);
    const int64_t id_base = *a.game_count;
    int64_t running = 0;
    for (int t = 0; t < tiles; ++t) {
        running += apply_tile<kRng>(a, t, running, id_base, warp_tot);
        __syncthreads();  // warp_tot is reused by the next tile
    }
    if (threadIdx.x == 0) {
        *a.game_count = id_base + running;
        *a.reset_count = running;
    }
}

// Large batches: the whole auto-reset in ONE cooperative launch.  A grid that fits the GPU in a single wave splits the
// slots into contiguous ranges, one per block, and every thread owns a run of consecutive 16-slot groups of it.
// Phase 1: the thread reads the `terminated` flags of its groups ONCE (all loads in flight together), keeps them as bit
// masks in shared memory, clears them in HBM; the block publishes how many of its games are over.  One grid-wide
// barrier.  Phase 2: every block sums the counts of the blocks before it (= the slot-ordered rank of its first finished
// game), lists its finished games in slot order in shared memory (one block scan) and resets them with CONVERGENT lanes
// (thread j takes list entry j) instead of one or two live lanes per warp walking a 512-slot stretch; the one-hot rows
// of the reset games are then written by all threads of the block from the boards parked in shared memory.
// Measured at M = 2^24, steady state (0.93 % of the games over), tools/prepare_probe.py with a cold L2: 65 us against
// 68.7 us for count + scan + apply; in the rollout loop 55 against 60 us (93 against 96 us with the fp32 one-hot rows).
// Launch + phase 1 + barrier are 15 us of that; the rest is the scattered stores of the 156 000 reset games themselves
// (eight arrays, one partly written 32-byte sector each), which the three-launch path pays as well.
constexpr int kFusedGroupsPerThread = 32;                             // at most
constexpr int kFusedMaxGroups = kPrepThreads * kFusedGroupsPerThread;  // 16-slot groups per block (masks: 16 KiB)
constexpr int kFusedListCap = 1024;                                    // finished games reset per pass

// all threads of the block write the one-hot rows of `n` games whose boards and slots are in shared memory
template <int kDtype>
__device__ __forceinline__ void write_onehot_listed(const uint4 *boards, const uint32_t *slots, int n, void *out_base)
{
    using P = OneHotPiece<kDtype>;
    constexpr int kPer = P::kPiecesPerGame;
    constexpr int kGamesPerPass = kPrepThreads / kPer;
    typename P::vec *out = reinterpret_cast<typename P::vec *>(out_base);
    const int piece = threadIdx.x % kPer;
    for (int j = threadIdx.x / kPer; j < n; j += kGamesPerPass)
        store_streaming(out + (int64_t)slots[j] * kPer + piece, P::make(boards, j, piece));
}

template <int kRng>
__global__ void __launch_bounds__(kPrepThreads, 5) prepare_fused_kernel(const ml2048_prepare_args a, int32_t *block_counts)
{
    cg::grid_group grid = cg::this_grid();
    __shared__ uint16_t s_mask[kFusedMaxGroups];
    __shared__ uint32_t s_list[kFusedListCap];
    __shared__ uint4 s_board[kFusedListCap];
    __shared__ int warp_tot[kPrepThreads / 32];
    const int64_t n16 = (a.num_games + 15) / 16;
    const int64_t per_block = (n16 + gridDim.x - 1) / gridDim.x;
    const int64_t begin = (int64_t)blockIdx.x * per_block;
    const int64_t end = begin + per_block < n16 ? begin + per_block : n16;
    const int groups = end > begin ? (int)(end - begin) : 0;
    const int per_thread = (int)((per_block + kPrepThreads - 1) / kPrepThreads);  // <= kFusedGroupsPerThread
    const int k_first = threadIdx.x * per_thread;
    const int k_last = k_first + per_thread < groups ? k_first + per_thread : groups;  // this thread owns [k_first, k_last)
    const int64_t id_base = *a.game_count;  // read before the barrier; block 0 advances it after the barrier

    // phase 1: flags -> masks in shared memory, flags cleared (entry.fill(0), game_numba.py:638-639), block count.
    // A thread's groups are adjacent (16 bytes each), so a warp's loads cover one dense stretch; four at a time
    int mine = 0;
    for (int k0 = k_first; k0 < k_last; k0 += 4) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
            v[u] = k0 + u < k_last ? reinterpret_cast<const uint4 *>(a.terminated)[begin + k0 + u] : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (k0 + u < k_last) {
                const uint32_t m = flags16(v[u]);
                s_mask[k0 + u] = (uint16_t)m;
                mine += __popc(m);
                if (m) reinterpret_cast<uint4 *>(a.terminated)[begin + k0 + u] = make_uint4(0, 0, 0, 0);
            }
        }
    }
    // the block's count, and the rank of this thread's first finished game inside the block (phase 2)
    const BlockScan in_block = block_scan<kPrepThreads>(mine, warp_tot);
    const int block_total = in_block.total, my_first = in_block.below;
    if (threadIdx.x == 0) block_counts[blockIdx.x] = block_total;
    grid.sync();

    // finished games in the blocks before this one, and in all blocks
    int before = 0, all = 0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += kPrepThreads) {
        const int c = block_counts[b];
        all += c;
        before += b < (int)blockIdx.x ? c : 0;
    }
    __syncthreads();
    before = block_scan<kPrepThreads>(before, warp_tot).total;
    __syncthreads();
    all = block_scan<kPrepThreads>(all, warp_tot).total;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        *a.game_count = id_base + all;
        *a.reset_count = all;
    }
    if (block_total == 0) return;

    // phase 2: list this block's finished games in slot order and reset them
    const PrepDraws draws = prep_draws(a, a.philox_counter, a.sched != nullptr);
    // passes of kFusedListCap games (one pass unless a large share of the block's games is over, e.g. right after reset())
    for (int window = 0; window < block_total; window += kFusedListCap) {
        const int n = block_total - window < kFusedListCap ? block_total - window : kFusedListCap;
        if (my_first < window + n && my_first + mine > window) {  // some of this thread's games fall into the window
            int p = my_first - window;
            for (int k = k_first; k < k_last; ++k) {
                uint32_t m = s_mask[k];
                const uint32_t g0 = (uint32_t)((begin + k) * 16);
                while (m) {
                    if (p >= 0 && p < n) s_list[p] = g0 + (uint32_t)(__ffs((int)m) - 1);
                    ++p;
                    m &= m - 1u;
                }
            }
        }
        __syncthreads();  // the list is complete
        for (int j = threadIdx.x; j < n; j += kPrepThreads)
            s_board[j] = reset_slot<kRng>(a, draws, s_list[j], (int64_t)before + window + j, id_base);
        if (a.onehot) {
            __syncthreads();  // the boards are parked
            with_onehot_dtype(a.onehot_dtype, [&](auto k) { write_onehot_listed<decltype(k)::value>(s_board, s_list, n, a.onehot); });
        }
        __syncthreads();  // list and boards may be overwritten
    }
}

// ---- fused auto-reset: bookkeeping kernels ----------------------------------------------------

constexpr int kScanThreads = 1024;  // groups per chunk

// One launch over the `terminated` flags (1 byte per game, the authoritative record of which games are over): thread i
// counts the finished games of slots [32i, 32i+32) (two 16-byte loads), every block scans its chunk of 1024 such group counts
// (reset_rank = exclusive prefix inside the chunk) and posts the chunk total; the block that finishes LAST (ticket) scans the chunk totals into reset_chunk_base and advances the id counter.
// scratch: [0, chunks) chunk totals, [chunks] ticket (zero between launches), [chunks + 1] unused.
__global__ void __launch_bounds__(kScanThreads) autoreset_scan_kernel(const uint4 *term16, int64_t n16, int32_t *reset_rank,
                                                                      int32_t *reset_chunk_base, int64_t groups, int64_t *game_count,
                                                                      const int64_t *id_offset, int64_t *reset_id_base,
                                                                      int64_t *reset_count, int32_t *scratch)
{
    __shared__ int warp_tot[kScanThreads / 32];
    __shared__ bool last_s;
    // Programmatic dependent launch: the fused step that follows may start (load its boards, which the PREVIOUS step wrote and
    // this kernel does not touch) as soon as every block of this scan is running; it waits (griddepcontrol.wait) before it reads
    // what the scan writes or writes what the scan reads.
    asm volatile("griddepcontrol.launch_dependents;");
    const int chunks = (int)gridDim.x;
    const int64_t i = (int64_t)blockIdx.x * kScanThreads + threadIdx.x;
    int v = 0;
    if (i < groups) {
        v = __popc(flags16(term16[2 * i]));
        if (2 * i + 1 < n16) v += __popc(flags16(term16[2 * i + 1]));  // the padding stops at a multiple of 16 flags
    }
    const BlockScan s = block_scan<kScanThreads>(v, warp_tot);
    if (i < groups) reset_rank[i] = s.below;
    if (threadIdx.x == 0) {
        scratch[blockIdx.x] = s.total;
        __threadfence();
        last_s = atomicAdd(&scratch[chunks], 1) == chunks - 1;
    }
    __syncthreads();
    if (!last_s) return;
    // the last block: exclusive scan over the chunk totals (volatile reads: they were written by other blocks)
    __threadfence();
    const int total = block_scan_passes<kScanThreads>(scratch, reset_chunk_base, chunks, warp_tot);
    if (threadIdx.x == 0) {
        const int64_t base = *game_count + (id_offset ? *id_offset : 0);
        *reset_id_base = base;
        if (!id_offset) *game_count = base + total;
        *reset_count = total;
        scratch[chunks] = 0;  // ticket for the next launch
    }
}

// ---- small stand-alone ops ------------------------------------------------------------------

template <int kDtype>
__global__ void __launch_bounds__(kStepThreads) onehot_kernel(const uint4 *boards, void *out, int64_t num_games)
{
    __shared__ uint4 sboards[kStepThreads];
    const int64_t block_first = (int64_t)blockIdx.x * kStepThreads;
    const int64_t g = block_first + threadIdx.x;
    sboards[threadIdx.x] = (g < num_games) ? boards[g] : make_uint4(0, 0, 0, 0);
    __syncthreads();
    const int64_t remaining = num_games - block_first;
    write_onehot_tile<kDtype, kStepThreads>(sboards, remaining < kStepThreads ? (int)remaining : kStepThreads, out, block_first);
}

__global__ void __launch_bounds__(kStepThreads) valid_kernel(const uint4 *boards, uint32_t *valid, int64_t num_games)
{
    const int64_t g = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    if (g >= num_games) return;
    const uint4 b = boards[g];
    valid[g] = valid_mask(b.x, b.y, b.z, b.w);
}

__global__ void __launch_bounds__(kStepThreads) max_tile_hist_kernel(const uint4 *boards, const uint8_t *terminated,
                                                                     int64_t num_games, unsigned long long *hist20)
{
    __shared__ unsigned int sh[20];
    if (threadIdx.x < 20) sh[threadIdx.x] = 0u;
    __syncthreads();
    for (int64_t g = (int64_t)blockIdx.x * kStepThreads + threadIdx.x; g < num_games; g += (int64_t)gridDim.x * kStepThreads) {
        if (terminated && !terminated[g]) continue;
        const uint4 b = boards[g];
        atomicAdd(&sh[min(max_cell(b.x, b.y, b.z, b.w), 19u)], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 20 && sh[threadIdx.x]) atomicAdd(&hist20[threadIdx.x], (unsigned long long)sh[threadIdx.x]);
}

__global__ void __launch_bounds__(kStepThreads) sample_random_valid_kernel(const uint32_t *valid, uint8_t *actions, int64_t num_games,
                                                                           int64_t slot_base, uint64_t seed, uint64_t counter)
{
    const int64_t g = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    if (g >= num_games) return;
    const uint64_t slot = (uint64_t)(slot_base + g);
    const uint32_t word = slot_word(slot, counter, seed, 0u);  // the same policy word the step kernel draws
    const uint32_t bits = mask_bits4(valid[g]);
    const uint32_t nv = popc32(bits);
    actions[g] = (uint8_t)(nv ? kth_valid_action(bits, umulhi32(word, nv)) : 0u);
}

__global__ void __launch_bounds__(kStepThreads) sample_categorical_kernel(const float4 *logits, const uint32_t *valid, uint8_t *act8,
                                                                          long long *act64, float *log_prob, int64_t num_games,
                                                                          int64_t slot_base, uint64_t seed, uint64_t counter)
{
    const int64_t g = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    if (g >= num_games) return;
    const uint64_t slot = (uint64_t)(slot_base + g);
    const uint32_t word = slot_word(slot, counter, seed, 0u);  // the same policy word the step kernel draws
    const uint32_t vm = valid[g];
    const uint32_t bits = ((vm & 0xffu) ? 1u : 0u) | ((vm & 0xff00u) ? 2u : 0u) | ((vm & 0xff0000u) ? 4u : 0u) | ((vm & 0xff000000u) ? 8u : 0u);
    const float4 lg = logits[g];
    float lp;
    const uint32_t action = sample_masked_categorical(lg.x, lg.y, lg.z, lg.w, bits, word, lp);
    if (act8) act8[g] = (uint8_t)action;
    if (act64) act64[g] = (long long)action;
    if (log_prob) log_prob[g] = lp;
}

// compute_gae's reverse scan (gae.py:50, :65-68).  Layout (use, step, game), game fastest: a warp reads 32
// adjacent games of one (use, step) row.  __fmul_rn/__fadd_rn keep the reference's rounding (no FMA contraction).
__global__ void __launch_bounds__(kStepThreads) gae_kernel(const float *v0, const float *v1, const float *reward,
                                                           const uint8_t *terminated, float *adv, int64_t step_count,
                                                           int64_t game_count, int64_t total, float gamma, float coef)
{
    const int64_t i = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;  // over use x game
    if (i >= total) return;
    const int64_t u = i / game_count, g = i - u * game_count;
    const int64_t base = u * step_count * game_count + g;
    float tmp = 0.0f;
    // the loads do not depend on the running value: fetch eight steps at a time so that many rows are in flight
    // (measured at (2, 64, 2^20): 2 ahead 890 us, 4 ahead 418 us, 8 ahead 357 us = 6.39 TB/s, 16 ahead 359 us)
    int64_t t = step_count - 1;
#ifndef ML2048_GAE_AHEAD
#define ML2048_GAE_AHEAD 8
#endif
    constexpr int kAhead = ML2048_GAE_AHEAD;
    for (; t >= kAhead - 1; t -= kAhead) {
        float a0[kAhead], a1[kAhead], rw[kAhead], mk[kAhead];
#pragma unroll
        for (int j = 0; j < kAhead; ++j) {
            const int64_t k = base + (t - j) * game_count;
            a0[j] = v0[k], a1[j] = v1[k], rw[j] = reward[k], mk[j] = terminated[k] ? 0.0f : 1.0f;
        }
#pragma unroll
        for (int j = 0; j < kAhead; ++j) {
            // delta = gamma * v1 * mask + reward - v0, evaluated left to right in fp32
            const float delta = __fsub_rn(__fadd_rn(__fmul_rn(__fmul_rn(gamma, a1[j]), mk[j]), rw[j]), a0[j]);
            tmp = __fmul_rn(tmp, coef);
            tmp = __fadd_rn(delta, __fmul_rn(tmp, mk[j]));
            adv[base + (t - j) * game_count] = tmp;
        }
    }
    for (; t >= 0; --t) {
        const int64_t k = base + t * game_count;
        const float mask = terminated[k] ? 0.0f : 1.0f;
        const float delta = __fsub_rn(__fadd_rn(__fmul_rn(__fmul_rn(gamma, v1[k]), mask), reward[k]), v0[k]);
        tmp = __fmul_rn(tmp, coef);
        tmp = __fadd_rn(delta, __fmul_rn(tmp, mask));
        adv[k] = tmp;
    }
}

// The flags a host caller reads after a step -- valid_actions (four 0/1 bytes), terminated, invalid -- as ONE byte per game for
// the trip over PCIe: bits 0..3 = left, right, up, down valid, bit 4 = terminated, bit 5 = invalid.  Four games per thread.
__global__ void __launch_bounds__(kStepThreads) pack_flags_kernel(const uint32_t *valid, const uint8_t *terminated, const uint8_t *invalid,
                                                                  uint8_t *packed, int64_t num_games)
{
    const int64_t g = ((int64_t)blockIdx.x * kStepThreads + threadIdx.x) * 4;
    if (g >= num_games) return;
    const bool whole = g + 4 <= num_games && ((reinterpret_cast<uintptr_t>(valid) & 15u) | (reinterpret_cast<uintptr_t>(packed) & 3u) |
                                               (reinterpret_cast<uintptr_t>(terminated) & 3u) | (reinterpret_cast<uintptr_t>(invalid) & 3u)) == 0u;
    if (whole) {
        const uint4 v = *reinterpret_cast<const uint4 *>(valid + g);
        uint32_t out = mask_bits4(v.x) | (mask_bits4(v.y) << 8) | (mask_bits4(v.z) << 16) | (mask_bits4(v.w) << 24);
        if (terminated) out |= (*reinterpret_cast<const uint32_t *>(terminated + g) & 0x01010101u) << 4;
        if (invalid) out |= (*reinterpret_cast<const uint32_t *>(invalid + g) & 0x01010101u) << 5;
        *reinterpret_cast<uint32_t *>(packed + g) = out;
    } else {
        for (int64_t i = g; i < num_games && i < g + 4; ++i)
            packed[i] = (uint8_t)(mask_bits4(valid[i]) | (terminated ? (terminated[i] & 1u) << 4 : 0u) | (invalid ? (invalid[i] & 1u) << 5 : 0u));
    }
}

__global__ void fill_terminated_kernel(uint8_t *terminated, int64_t num_games, int64_t padded)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < padded) terminated[i] = (i < num_games) ? 1 : 0;
}

// ---- afterstates ----------------------------------------------------------------------------
// The four moves of every board without the spawn: what step(a) computes up to game_numba.py:728, for every a.  One thread per
// (game, direction): thread t = 4 * game + direction, so the four lanes of a game read the same 16-byte board (one L1 sector)
// and every output is indexed by t -- a warp stores 512 contiguous bytes of boards, 128 of rewards, 32 of flags, 512 of
// `merged`.  The move, the reward and the `merged` log are the step kernel's own functions (move_board_sel with a row of
// d_move_sel, step_reward, fusion_log).  A direction that does not change the board gets reward 0 (the step kernel leaves
// the stale reward there instead); it fuses nothing, so its `merged` row is 0 as well.

// Board `bd` moved in direction `dir` (0..3) without the spawn: the moved board in `now`, what fused in `f`; true iff the move
// changed the board, i.e. the direction is valid
__device__ __forceinline__ bool try_move(uint4 bd, uint32_t dir, uint4 &now, Fusions &f)
{
    uint32_t r0 = bd.x, r1 = bd.y, r2 = bd.z, r3 = bd.w;
    move_board_sel(r0, r1, r2, r3, d_move_sel + dir * kMoveSelRow, f);
    now = make_uint4(r0, r1, r2, r3);
    return ((r0 ^ bd.x) | (r1 ^ bd.y) | (r2 ^ bd.z) | (r3 ^ bd.w)) != 0u;
}

template <bool kLog>
__global__ void __launch_bounds__(kStepThreads) afterstates_kernel(const uint4 *board, uint4 *after, float *reward, uint8_t *valid,
                                                                   uint4 *merged, int32_t reward_kind, int64_t num_games)
{
    const int64_t t = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;  // 64-bit: 16 * t passes 2^31 at 2^25 games
    if (t >= 4 * num_games) return;
    const uint4 bd = board[t >> 2];
    uint4 now;
    Fusions f;
    const bool moved = try_move(bd, threadIdx.x & 3u, now, f);
    after[t] = now;
    reward[t] = moved ? step_reward<false>(reward_kind, f, now, bd, fusion_gain(f)) : 0.0f;
    valid[t] = moved ? 1 : 0;
    if (kLog) {
        uint32_t m0, m1, m2, m3;
        fusion_log(f, m0, m1, m2, m3);
        merged[t] = make_uint4(m0, m1, m2, m3);
    }
}

// ---- n-tuple networks -----------------------------------------------------------------------
// Value, greedy afterstate move and TD(0) update of an n-tuple network (board_ops.cuh: NTupleSpec, ntuple_value).  The spec is
// a by-value __grid_constant__ parameter: the kernels index it in the constant bank, nothing is copied to local memory.
// Board offsets are 64-bit (16 * game passes 2^31 at 2^27 games); table entry indices stay below 2^28.
// Every n-tuple kernel below is a template over the spec: Spec = NTupleSpec is the single-stage network, Spec =
// NTupleStagedSpec the multi-stage one (board_ops.cuh: one weight set per stage, stage(b) = #{k : tau_k <= max_c min(b[c], 15)},
// stage s's tables at s * N; indices below 8 * 2^28).  The staged visitor adds stage(b) * N to every offset it reports, so
// a board's value, greedy's afterstates, expectimax's leaves and the lambda window's boards each use their own stage's tables,
// and the updates (scatter, TC accumulate and apply, whose claim is on j = off + idx) write the entries of x_0's stage.  One
// stage launches the NTupleSpec instances (with_spec below).

// one thread per board
template <class Spec>
__global__ void __launch_bounds__(kStepThreads) ntuple_value_kernel(const uint4 *board, const float *w, __grid_constant__ const Spec spec,
                                                                    float *value, int64_t num_games)
{
    const int64_t i = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    if (i >= num_games) return;
    const uint4 b = board[i];
    value[i] = ntuple_value(w, spec, ntuple_nibbles(b.x, b.y, b.z, b.w));
}

// One thread per (board, direction), thread t = 4 * game + direction as in afterstates_kernel: the move, its reward and its
// validity are the step kernel's own (move_board_sel, step_reward), the afterstate's value is looked up in registers and the
// four lanes pick the move with a shuffle argmax -- no afterstate goes to memory.  q = reward + V(afterstate) for a direction
// that changes the board; NaN ranks as -inf; the largest q wins, ties go to the smallest direction.  A board without a valid
// direction gets action 0 and its own board, reward 0, value 0.  The lane of the chosen direction writes the outputs.
template <class Spec>
__global__ void __launch_bounds__(kStepThreads) ntuple_greedy_kernel(const uint4 *board, const float *w, __grid_constant__ const Spec spec,
                                                                     int32_t reward_kind, uint8_t *action_u8, long long *action_i64,
                                                                     uint4 *after, float *reward, float *value, int64_t num_games)
{
    const int64_t t = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    const bool live = t < 4 * num_games;  // all four lanes of a game are live or none: the shuffles below need every lane
    const uint32_t a = threadIdx.x & 3u;
    const uint4 bd = live ? board[t >> 2] : make_uint4(0u, 0u, 0u, 0u);
    uint4 now;
    Fusions f;
    const bool moved = try_move(bd, a, now, f);
    float r = 0.0f, v = 0.0f, key = -INFINITY;
    if (moved) {
        r = step_reward<false>(reward_kind, f, now, bd, fusion_gain(f));
        v = ntuple_value(w, spec, ntuple_nibbles(now.x, now.y, now.z, now.w));
        const float q = r + v;
        key = (q == q) ? q : -INFINITY;
    }
    // (valid, key) descending, then direction ascending: a total order, so both butterfly steps leave every lane with the winner
    uint32_t code = a | (moved ? 4u : 0u);
#pragma unroll
    for (int m = 1; m <= 2; m <<= 1) {
        const float okey = __shfl_xor_sync(0xffffffffu, key, m);
        const uint32_t ocode = __shfl_xor_sync(0xffffffffu, code, m);
        const bool ovalid = (ocode & 4u) != 0u, valid = (code & 4u) != 0u;
        if (ovalid && (!valid || okey > key || (okey == key && (ocode & 3u) < (code & 3u)))) key = okey, code = ocode;
    }
    const uint32_t chosen = (code & 4u) ? (code & 3u) : 0u;
    if (!live || a != chosen) return;
    const int64_t g = t >> 2;
    if (action_u8) action_u8[g] = (uint8_t)a;
    else action_i64[g] = (long long)a;
    after[g] = now;  // == bd when no direction is valid (direction 0 then leaves the board as it is)
    reward[g] = r;
    value[g] = v;
}

// TD(0), phase 1: delta = alpha * (target - V(afterstate)) for every masked-in game with the weights as they were before the
// update (phase 2 runs as a second launch); 0 for a masked-out game
template <class Spec>
__global__ void __launch_bounds__(kStepThreads) ntuple_td_delta_kernel(const uint4 *after, const float *target, const uint8_t *mask, float alpha,
                                                                       const float *w, __grid_constant__ const Spec spec, float *delta,
                                                                       int64_t num_games)
{
    const int64_t i = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    if (i >= num_games) return;
    float d = 0.0f;
    if (!mask || mask[i]) {
        const uint4 b = after[i];
        d = alpha * (target[i] - ntuple_value(w, spec, ntuple_nibbles(b.x, b.y, b.z, b.w)));
    }
    delta[i] = d;
}

// TD(0), phase 2: w[entry] += delta for every masked-in game, tuple and image.  Float atomics (RED.ADD.F32): the order of the
// adds that different games make to one entry is unspecified, so the weights are reproducible up to the fp32 rounding of
// that order.
template <class Spec>
__global__ void __launch_bounds__(kStepThreads) ntuple_td_scatter_kernel(const uint4 *after, const uint8_t *mask, const float *delta, float *w,
                                                                         __grid_constant__ const Spec spec, int64_t num_games)
{
    const int64_t i = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    if (i >= num_games || (mask && !mask[i])) return;
    const uint4 b = after[i];
    const float d = delta[i];
    ntuple_for_each_entry(spec, ntuple_nibbles(b.x, b.y, b.z, b.w), [&](uint32_t off, uint32_t idx) { atomicAdd(w + off + idx, d); });
}

// ---- temporal coherence (TC) learning ---------------------------------------------------------
// Definition (ml2048_tc_update in the header, ops.ntuple_tc_update and tests/_tc_ref.py say the same; every operation is one
// float32 operation, __fmul_rn / __fadd_rn / __fdiv_rn, no contraction).  C[j] = {E_j, A_j}: the running sum of the errors
// applied to entry j and of their absolute values.  One synchronous batch:
//   1. delta_i = alpha * (target_i - V(after_i)) with the weights before the call, 0 for a masked-out game (phase 1 is
//      ntuple_td_delta_kernel: TD(0)'s delta bit for bit);
//   2. for every masked-in game and each of its 8K entries j (twice if the game hits j twice): dE_j += delta_i,
//      dA_j += |delta_i| (float atomics: order within one entry unspecified, subnormals flushed);
//   3. for every entry with dA_j != 0 (NaN counts as non-zero), with E_j, A_j as they were before the call:
//      beta_j = (A_j == 0) ? 1 : |E_j| / A_j;  w_j += beta_j * dE_j;  E_j += dE_j;  A_j += dA_j.
//      Entries with dA_j == 0 stay as they are, bit for bit.
// E and A sum alpha-scaled errors: with a constant alpha beta is the unscaled rule's, a changing alpha weights older errors
// by the alpha they had.  The accumulator acc[j] = {dE_j, dA_j} belongs to the caller and is all zero bits on entry and on
// return.  Cost O(batch): phase 3 walks the batch's own entries, never the table.

// TC, phase 2: one 8-byte vector atomic (RED.E.ADD.F32x2) per lookup into the interleaved {dE, dA} accumulator
template <class Spec>
__global__ void __launch_bounds__(kStepThreads) ntuple_tc_accumulate_kernel(const uint4 *after, const uint8_t *mask, const float *delta,
                                                                            float2 *acc, __grid_constant__ const Spec spec,
                                                                            int64_t num_games)
{
    const int64_t i = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    if (i >= num_games || (mask && !mask[i])) return;
    const uint4 b = after[i];
    const float d = delta[i];
    const float2 e = make_float2(d, fabsf(d));
    ntuple_for_each_entry(spec, ntuple_nibbles(b.x, b.y, b.z, b.w), [&](uint32_t off, uint32_t idx) { atomicAdd(acc + off + idx, e); });
}

// TC, phase 3: one thread per masked-in game walks its own entries and claims each with a 64-bit exchange against 0; only
// the thread that receives dA != 0 applies the entry, with plain loads and stores (no other thread touches w[j] or C[j] in
// this launch).  So every accumulated entry is applied exactly once and the accumulator is zero again afterwards.  A plain
// L2 load first skips the exchange where the word is already zero (an entry claimed by an earlier game: early-game entries are
// shared by thousands of games): the word only goes from non-zero to zero during this launch, so a zero read is final and a
// stale non-zero read costs one exchange that returns 0.  The whole word is tested, not only dA, so that a -0 left in dE is
// still cleared.  -DML2048_TC_APPLY_ALWAYS_EXCHANGE builds the variant without the load (tools/tc_bench.py times both).
template <class Spec>
__global__ void __launch_bounds__(kStepThreads) ntuple_tc_apply_kernel(const uint4 *after, const uint8_t *mask, float *w, float2 *coh,
                                                                       unsigned long long *acc, __grid_constant__ const Spec spec,
                                                                       int64_t num_games)
{
    const int64_t i = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    if (i >= num_games || (mask && !mask[i])) return;
    const uint4 b = after[i];
    ntuple_for_each_entry(spec, ntuple_nibbles(b.x, b.y, b.z, b.w), [&](uint32_t off, uint32_t idx) {
        const uint32_t j = off + idx;
#if !defined(ML2048_TC_APPLY_ALWAYS_EXCHANGE)
        if (__ldcg(acc + j) == 0ull) return;
#endif
        const unsigned long long word = atomicExch(acc + j, 0ull);
        const float dE = __uint_as_float((uint32_t)word), dA = __uint_as_float((uint32_t)(word >> 32));
        if (dA == 0.0f) return;  // NaN goes on
        const float2 c = coh[j];
        const float beta = c.y == 0.0f ? 1.0f : __fdiv_rn(fabsf(c.x), c.y);
        w[j] = __fadd_rn(w[j], __fmul_rn(beta, dE));
        coh[j] = make_float2(__fadd_rn(c.x, dE), __fadd_rn(c.y, dA));
    });
}

// ---- weight promotion (board_ops.cuh: NTuplePromotedSpec) ------------------------------------------
// The reads and the delta phases of a promoting network are the kernels of this file instantiated with NTuplePromotedSpec:
// only ntuple_value differs, and it reads the marks with __ldg because no read launch writes them.  An update then runs this
// promote phase between its delta and apply launches on the same stream, and applies with the staged kernels, which write
// the entries of x_0's own stage.  `mark_words` = the marks as 32-bit words.

// Mark byte e, read with an acquire load of its whole 32-bit word (the size the atomicOr below writes): the weight and
// coherence stores of the thread that set a bit seen here are visible after it
__device__ __forceinline__ uint32_t load_mark_acquire(const uint32_t *words, uint32_t e)
{
    uint32_t m;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(m) : "l"(words + (e >> 2)) : "memory");
    return (m >> (8u * (e & 3u))) & 0xffu;
}

// One thread per masked-in game with x_0 in stage s0 >= 1 walks x_0's entries e; where the mark of (s0, e) is clear it
// stores w[s0 * N + e] = W(s0 - 1, e) (and TC's coherence {0, 0}), then __threadfence() and an atomicOr of the bit into the
// mark's 32-bit word (release).  Two games of one launch can meet the same e in different stages, so a game at stage s0 may
// find the mark of a lower stage k being set while it reads.  It reads marks with acquire loads and weights with L2 loads
// (__ldcg, not the read-only path), so it sees either the bit clear, and reads a lower source whose storage this launch
// does not write, or the bit set, and reads the copy that bit publishes.  Either way it gets W_before(k, e): stage k's copy
// is W_before(k - 1, e) = W_before(k, e) when its mark was clear before the call, and untouched when it was set.  So every
// writer of an entry stores the same value, no add happens in this launch, and the result does not depend on the order.
// Stage 0 is never written here.
__global__ void __launch_bounds__(kStepThreads) ntuple_promote_kernel(const uint4 *after, const uint8_t *mask, float *w, float2 *coh,
                                                                      uint32_t *mark_words, __grid_constant__ const NTupleStagedSpec spec,
                                                                      int64_t num_games)
{
    const int64_t i = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    if (i >= num_games || (mask && !mask[i])) return;
    const uint4 b = after[i];
    const uint64_t nib = ntuple_nibbles(b.x, b.y, b.z, b.w);
    const uint32_t s0 = ntuple_stage(spec, nib);
    if (s0 == 0u) return;
    const uint32_t bit = 1u << (s0 - 1u), n = spec.stage_size;
    ntuple_for_each_entry(static_cast<const NTupleSpec &>(spec), nib, [&](uint32_t off, uint32_t idx) {
        const uint32_t e = off + idx;
        const uint32_t m = load_mark_acquire(mark_words, e);
        if (m & bit) return;
        w[s0 * n + e] = __ldcg(w + ntuple_source_stage(s0, m) * n + e);
        if (coh) coh[s0 * n + e] = make_float2(0.0f, 0.0f);
        __threadfence();
        atomicOr(mark_words + (e >> 2), bit << (8u * (e & 3u)));
    });
}

// ---- delayed TD(lambda) / TC(lambda) ------------------------------------------------------------
// Definition (ml2048_lambda_td_update in the header, ops.ntuple_td_lambda_update and tests/_lambda_ref.py say the same; every
// operation is one float32 operation, __fadd_rn / __fmul_rn, no contraction).  Game i's window is x_0 ... x_h: x_0 the
// afterstate being updated (chosen h learner steps ago), x_h the one chosen this step; rho_k (k = 1..h) the reward of the move
// that produced x_k; e_k (k = 0..h-1) = 1 when the environment step after x_k was chosen ended the game; V_k = V(x_k) with the
// weights as they are before the call (ntuple_value).  With lf = float32(lambda) and c = 1.0f - lf rounded once on the host:
//   R_{h-1} = e_{h-1} ? 0 : rho_h + V_h
//   R_k     = e_k     ? 0 : (rho_{k+1} + c * V_{k+1}) + lf * R_{k+1}      for k = h-2 ... 0
//   delta   = alpha * (R_0 - V_0)                                         (0 for a masked-out game)
// h = 1 is TD(0)'s delta bit for bit.  Ring: after [h+1][M][16], reward [h+1][M], ended [h+1][M]; x_k is in slot
// (newest - (h - k)) mod (h + 1) = (newest + 1 + k) mod (h + 1); the ended byte of the newest slot is not read.  The update of
// x_0's entries is then TD(0)'s scatter or TC's phases 2 and 3 on x_0's slot, launched after this kernel: every delta is
// computed before any weight is written.

constexpr int kLambdaMaxHorizon = 16;

// one thread per game: the first end in the window fixes where the recursion starts, so the values after it are never
// looked up (they would be multiplied away by the 0 anyway, and skipping them changes no bit)
template <class Spec>
__global__ void __launch_bounds__(kStepThreads) ntuple_lambda_delta_kernel(const uint4 *after, const float *reward, const uint8_t *ended,
                                                                           const uint8_t *mask, int32_t horizon, int32_t newest, float lf,
                                                                           float c, float alpha, const float *w,
                                                                           __grid_constant__ const Spec spec, float *delta,
                                                                           int64_t num_games)
{
    const int64_t i = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    if (i >= num_games) return;
    float d = 0.0f;
    if (!mask || mask[i]) {
        const int32_t slots = horizon + 1;
        int32_t s0 = newest + 1;  // slot of x_0
        if (s0 == slots) s0 = 0;
        auto slot = [&](int32_t k) { const int32_t s = s0 + k; return s >= slots ? s - slots : s; };
        auto val = [&](int32_t k) {
            const uint4 b = after[(int64_t)slot(k) * num_games + i];
            return ntuple_value(w, spec, ntuple_nibbles(b.x, b.y, b.z, b.w));
        };
        int32_t top = horizon - 1;  // the first k with e_k = 1 (R_top = 0), else h - 1 (R_top = rho_h + V_h)
        bool end = false;
        for (int32_t k = 0; k < horizon && !end; ++k)
            if (ended[(int64_t)slot(k) * num_games + i]) top = k, end = true;
        float r = end ? 0.0f : __fadd_rn(reward[(int64_t)slot(horizon) * num_games + i], val(horizon));
        for (int32_t k = top - 1; k >= 0; --k)
            r = __fadd_rn(__fadd_rn(reward[(int64_t)slot(k + 1) * num_games + i], __fmul_rn(c, val(k + 1))), __fmul_rn(lf, r));
        d = __fmul_rn(alpha, __fsub_rn(r, val(0)));
    }
    delta[i] = d;
}

// ---- expectimax over an n-tuple network -----------------------------------------------------
// Definition (tests/_expectimax_ref.py is the same in NumPy; every operation is one float32 operation rounded on its own, so
// the sums and products below are __fadd_rn / __fmul_rn / __fdiv_rn and nvcc cannot contract them into FMAs).  after(b,a),
// r(b,a), valid(b,a) are afterstates_kernel's (the step kernel's move_board_sel and step_reward); V is ntuple_value;
// p2 = float32(two_prob), p4 = 1.0f - p2, both rounded on the host.
//   E(s, d), s an afterstate (>= 1 empty cell: a move that changed the board leaves one), d >= 1 chance layers left:
//       for every empty cell c of s in ascending order, t_c = p2 * M(s + tile 2 at c, d) + p4 * M(s + tile 4 at c, d); an
//       outcome of probability 0 is not evaluated (t_c = p2 * m2 when p4 == 0, p4 * m4 when p2 == 0);
//       S = t_c1 + t_c2 + ... added in that order from the first term (not from 0.0f: signed zeros survive); E = S / n.
//   M(b, d) = max over the valid a of key(r(b,a) + (d == 1 ? V(after(b,a)) : E(after(b,a), d - 1))), key(NaN) = -inf; among
//       equal keys the smallest direction's key is taken (ntuple_greedy's tie rule); 0 for a board without a valid move.
//   Root, depth D in {1, 2}: q_a = r(b,a) + E(after(b,a), D) for a valid a, -inf otherwise; the action is ntuple_greedy's
//       argmax of q (NaN as -inf, ties to the smallest direction); value = E(after(b,a*), D).  A board without a valid move:
//       action 0, its own board, reward 0, value 0, q all -inf.
// The spawn model is VecGame's marginal law: a uniform empty cell, a 2 with probability two_prob.  (VecGame ties 2-vs-4 to
// the cell for a table epoch; the search does not model that tie.)  No intermediate board leaves the registers.

// ntuple_greedy_kernel's 4-lane argmax (kept inline there: as a call it compiles to different SASS): lanes 4i..4i+3 hold
// direction code & 3, bit 2 of code = valid.  (valid, key) descending, then direction ascending is a total order, so both
// butterfly steps leave every lane of the group with the winner's key and code.
__device__ __forceinline__ void lane4_argmax(float &key, uint32_t &code)
{
#pragma unroll
    for (int m = 1; m <= 2; m <<= 1) {
        const float okey = __shfl_xor_sync(0xffffffffu, key, m);
        const uint32_t ocode = __shfl_xor_sync(0xffffffffu, code, m);
        const bool ovalid = (ocode & 4u) != 0u, valid = (code & 4u) != 0u;
        if (ovalid && (!valid || okey > key || (okey == key && (ocode & 3u) < (code & 3u)))) key = okey, code = ocode;
    }
}

// 16-bit mask of the empty cells of a board
__device__ __forceinline__ uint32_t empty_cells(uint4 s)
{
    return empties16(~occupied_signs(s.x) & kHi, ~occupied_signs(s.y) & kHi, ~occupied_signs(s.z) & kHi, ~occupied_signs(s.w) & kHi);
}

// The spawn outcomes of a chance node in evaluation order: outcome o is the (o / per_cell)-th empty cell with tile
// exponent 1 + (o & 1) when both tiles have a non-zero probability (per_cell = 2), else the one tile that has.
struct SpawnLaw {
    float p2, p4;
    __device__ __forceinline__ uint32_t per_cell() const { return (p2 > 0.0f && p4 > 0.0f) ? 2u : 1u; }
    __device__ __forceinline__ uint32_t tile(uint32_t o) const { return per_cell() == 2u ? 1u + (o & 1u) : (p2 > 0.0f ? 1u : 2u); }
};

// E(s, 1) of an afterstate s that the whole warp holds (warp-uniform call; n >= 1 empty cells).  A pass covers 8 outcomes x
// 4 inner directions: lane = 4 * outcome + direction, the move, reward and value in registers, M by lane4_argmax.  Every
// lane then reads the pass's 8 M values by shuffle and adds the terms in ascending cell order, so all lanes return E.
template <class Spec>
__device__ __forceinline__ float chance1(uint4 s, const float *w, const Spec &spec, int32_t reward_kind, SpawnLaw law)
{
    const uint32_t lane = threadIdx.x & 31u, a = lane & 3u;
    const uint32_t empties = empty_cells(s), n = popc32(empties);
    const uint32_t per_cell = law.per_cell(), outcomes = n * per_cell;
    const float p_one = law.p2 > 0.0f ? law.p2 : law.p4;
    float sum = 0.0f;
    for (uint32_t base = 0; base < outcomes; base += 8u) {
        const uint32_t o = base + (lane >> 2);
        const bool live = o < outcomes;
        uint32_t r0 = s.x, r1 = s.y, r2 = s.z, r3 = s.w;
        put_cell_shift(r0, r1, r2, r3, kth_set_bit16(empties, live ? o / per_cell : 0u), law.tile(o));
        const uint4 sp = make_uint4(r0, r1, r2, r3);
        Fusions f;  // try_move written out: as a call it compiles this function to different SASS
        move_board_sel(r0, r1, r2, r3, d_move_sel + a * kMoveSelRow, f);
        const bool moved = live && ((r0 ^ sp.x) | (r1 ^ sp.y) | (r2 ^ sp.z) | (r3 ^ sp.w)) != 0u;
        float key = -INFINITY;
        if (moved) {
            const float q = step_reward<false>(reward_kind, f, make_uint4(r0, r1, r2, r3), sp, fusion_gain(f)) +
                            ntuple_value(w, spec, ntuple_nibbles(r0, r1, r2, r3));
            key = (q == q) ? q : -INFINITY;
        }
        uint32_t code = a | (moved ? 4u : 0u);
        lane4_argmax(key, code);
        const float m = (code & 4u) ? key : 0.0f;  // M: 0 for a spawned board without a valid move
        if (per_cell == 2u) {
#pragma unroll
            for (uint32_t j = 0; j < 4u; ++j) {
                const float m2 = __shfl_sync(0xffffffffu, m, 8u * j), m4 = __shfl_sync(0xffffffffu, m, 8u * j + 4u);
                const float t = __fadd_rn(__fmul_rn(law.p2, m2), __fmul_rn(law.p4, m4));
                if (base + 2u * j < outcomes) sum = (base == 0u && j == 0u) ? t : __fadd_rn(sum, t);
            }
        } else {
#pragma unroll
            for (uint32_t j = 0; j < 8u; ++j) {
                const float t = __fmul_rn(p_one, __shfl_sync(0xffffffffu, m, 4u * j));
                if (base + j < outcomes) sum = (base == 0u && j == 0u) ? t : __fadd_rn(sum, t);
            }
        }
    }
    return __fdiv_rn(sum, (float)n);
}

// The root of lanes 4i..4i+3 (direction = lane & 3) of a board: q = r + e for a valid direction, lane4_argmax over q, the
// group's lanes write q, the chosen lane the rest.  `e` = E(after(bd, lane & 3), D) (ignored where that move is invalid);
// `store` is false for groups that hold no board.
__device__ __forceinline__ void expectimax_root(uint4 bd, float e, bool store, int64_t g, int32_t reward_kind, uint8_t *action_u8,
                                                long long *action_i64, uint4 *after, float *reward, float *value, float *q_out)
{
    const uint32_t a = threadIdx.x & 3u;
    uint4 now;
    Fusions f;
    const bool moved = try_move(bd, a, now, f);
    float r = 0.0f, q = -INFINITY, key = -INFINITY;
    if (moved) {
        r = step_reward<false>(reward_kind, f, now, bd, fusion_gain(f));
        q = __fadd_rn(r, e);
        key = (q == q) ? q : -INFINITY;
    }
    uint32_t code = a | (moved ? 4u : 0u);
    lane4_argmax(key, code);
    if (!store) return;
    q_out[4 * g + a] = q;
    const uint32_t chosen = (code & 4u) ? (code & 3u) : 0u;
    if (a != chosen) return;
    if (action_u8) action_u8[g] = (uint8_t)a;
    else action_i64[g] = (long long)a;
    after[g] = now;  // == bd when no direction is valid
    reward[g] = r;
    value[g] = moved ? e : 0.0f;
}

constexpr int kExpectimaxThreads = 256;

#if !defined(ML2048_EXPECTIMAX_WARP_PER_BOARD)
constexpr int kExpectimax1BoardsPerBlock = kExpectimaxThreads / 128;

// Depth 1, one warp per (board, root direction): warp w of a block takes board 2 * block + w / 4, direction w & 3, and
// computes E(after, 1) with chance1; lanes 0..7 of warp 0 then pick both boards' moves from shared memory.
template <class Spec>
__global__ void __launch_bounds__(kExpectimaxThreads) expectimax1_kernel(const uint4 *board, const float *w, __grid_constant__ const Spec spec,
                                                                         int32_t reward_kind, SpawnLaw law, uint8_t *action_u8,
                                                                         long long *action_i64, uint4 *after, float *reward,
                                                                         float *value, float *q_out, int64_t num_games)
{
    __shared__ float sh_e[kExpectimaxThreads / 32];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const int64_t g = (int64_t)blockIdx.x * kExpectimax1BoardsPerBlock + (warp >> 2);
    const bool live = g < num_games;
    const uint4 bd = live ? board[g] : make_uint4(0u, 0u, 0u, 0u);
    uint4 now;
    Fusions f;
    float e = 0.0f;
    if (try_move(bd, warp & 3u, now, f)) e = chance1(now, w, spec, reward_kind, law);  // warp-uniform
    if (lane == 0u) sh_e[warp] = e;
    __syncthreads();
    if (warp != 0u) return;
    const uint32_t slot = lane >> 2;  // the block's boards are slots 0 and 1; the other groups shuffle along
    const int64_t gs = (int64_t)blockIdx.x * kExpectimax1BoardsPerBlock + slot;
    const bool store = slot < (uint32_t)kExpectimax1BoardsPerBlock && gs < num_games;
    expectimax_root(store ? board[gs] : make_uint4(0u, 0u, 0u, 0u), store ? sh_e[lane] : 0.0f, store, gs, reward_kind, action_u8,
                    action_i64, after, reward, value, q_out);
}
#else
constexpr int kExpectimax1BoardsPerBlock = kExpectimaxThreads / 32;

// Depth 1, one warp per board (the alternative mapping; profiles/expectimax_bench.txt): the warp computes E(after(b,a), 1)
// for a = 0..3 in turn, lane group 0 picks the move.  No shared memory, no barrier.
template <class Spec>
__global__ void __launch_bounds__(kExpectimaxThreads) expectimax1_kernel(const uint4 *board, const float *w, __grid_constant__ const Spec spec,
                                                                         int32_t reward_kind, SpawnLaw law, uint8_t *action_u8,
                                                                         long long *action_i64, uint4 *after, float *reward,
                                                                         float *value, float *q_out, int64_t num_games)
{
    const int64_t g = (int64_t)blockIdx.x * kExpectimax1BoardsPerBlock + (threadIdx.x >> 5);
    if (g >= num_games) return;  // warp-uniform
    const uint4 bd = board[g];
    float mine = 0.0f;
    for (uint32_t a = 0; a < 4u; ++a) {
        uint4 now;
        Fusions f;
        if (!try_move(bd, a, now, f)) continue;
        const float e = chance1(now, w, spec, reward_kind, law);
        if ((threadIdx.x & 3u) == a) mine = e;
    }
    expectimax_root(bd, mine, (threadIdx.x & 31u) < 4u, g, reward_kind, action_u8, action_i64, after, reward, value, q_out);
}
#endif

// Depth 2, one block per board.  Its depth-1 chance nodes after(s', a') -- s' = after(b, a) + one spawn outcome o, a' an inner
// direction -- are numbered root direction-major, then outcome, then a' (at most 4 * 30 * 4 = 480); warp w evaluates nodes
// w, w + 8, ... with chance1 and stores key(r(s',a') + E(after(s',a'), 1)) and validity in shared memory.  Lane group 0 of warp
// 0 then folds them, in the definition's fixed order, into M, t_c, S and E for each root direction and picks the move.
constexpr int kExpectimax2Nodes = 4 * 2 * 15 * 4;

template <class Spec>
__global__ void __launch_bounds__(kExpectimaxThreads) expectimax2_kernel(const uint4 *board, const float *w, __grid_constant__ const Spec spec,
                                                                         int32_t reward_kind, SpawnLaw law, uint8_t *action_u8,
                                                                         long long *action_i64, uint4 *after, float *reward,
                                                                         float *value, float *q_out)
{
    __shared__ float sh_key[kExpectimax2Nodes];
    __shared__ uint8_t sh_ok[kExpectimax2Nodes];
    const int64_t g = blockIdx.x;
    const uint4 bd = board[g];
    const uint32_t per_cell = law.per_cell();
    uint32_t count[4];  // nodes under root direction a: 4 * outcomes of after(b, a), 0 for an invalid a
#pragma unroll
    for (uint32_t a = 0; a < 4u; ++a) {
        uint4 now;
        Fusions f;
        count[a] = try_move(bd, a, now, f) ? 4u * per_cell * popc32(empty_cells(now)) : 0u;
    }
    const uint32_t total = count[0] + count[1] + count[2] + count[3];
    for (uint32_t j = threadIdx.x >> 5; j < total; j += kExpectimaxThreads / 32) {
        uint32_t a = 0u, rem = j;
#pragma unroll
        for (uint32_t i = 0; i < 3u; ++i)
            if (a == i && rem >= count[i]) rem -= count[i], a = i + 1u;
        uint4 s, now;
        Fusions f;
        try_move(bd, a, s, f);  // a valid root direction: the others have no nodes
        const uint32_t o = rem >> 2, inner = rem & 3u;
        uint32_t r0 = s.x, r1 = s.y, r2 = s.z, r3 = s.w;
        put_cell_shift(r0, r1, r2, r3, kth_set_bit16(empty_cells(s), o / per_cell), law.tile(o));
        const uint4 sp = make_uint4(r0, r1, r2, r3);
        const bool moved = try_move(sp, inner, now, f);
        float key = -INFINITY;
        if (moved) {  // warp-uniform
            const float rr = step_reward<false>(reward_kind, f, now, sp, fusion_gain(f));
            const float q = __fadd_rn(rr, chance1(now, w, spec, reward_kind, law));
            key = (q == q) ? q : -INFINITY;
        }
        if ((threadIdx.x & 31u) == 0u) sh_key[j] = key, sh_ok[j] = moved ? 1 : 0;
    }
    __syncthreads();
    if (threadIdx.x >= 32u) return;
    // every lane group folds the nodes of its direction a = lane & 3 (groups 1..7 repeat group 0's work and store nothing)
    const uint32_t a = threadIdx.x & 3u;
    uint32_t start = 0u, nodes = 0u;
#pragma unroll
    for (uint32_t i = 0; i < 4u; ++i) {
        if (i < a) start += count[i];
        if (i == a) nodes = count[i];
    }
    float sum = 0.0f;
    for (uint32_t c = 0; c < nodes; c += 4u * per_cell) {  // one empty cell of after(b, a) per iteration, ascending
        float m[2];
#pragma unroll
        for (uint32_t t = 0; t < 2u; ++t) {
            const uint32_t base = start + c + 4u * t;
            float best = 0.0f;
            bool any = false;
            if (t < per_cell) {
#pragma unroll
                for (uint32_t i = 0; i < 4u; ++i) {
                    const float k = sh_key[base + i];
                    if (sh_ok[base + i] && (!any || k > best)) best = k, any = true;
                }
            }
            m[t] = best;  // 0 for a spawned board without a valid move
        }
        const float term = per_cell == 2u ? __fadd_rn(__fmul_rn(law.p2, m[0]), __fmul_rn(law.p4, m[1]))
                                          : __fmul_rn(law.p2 > 0.0f ? law.p2 : law.p4, m[0]);
        sum = c == 0u ? term : __fadd_rn(sum, term);
    }
    const float e = nodes ? __fdiv_rn(sum, (float)(nodes / (4u * per_cell))) : 0.0f;
    expectimax_root(bd, e, threadIdx.x < 4u, g, reward_kind, action_u8, action_i64, after, reward, value, q_out);
}

// ---- launch helpers -------------------------------------------------------------------------

inline bool misaligned(const void *p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) != 0; }

// `step` and `score` must be the two halves of one array of 8-byte {int32 step, float score} records
inline bool not_a_step_score_pair(const int32_t *step, const float *score)
{
    return misaligned(step, 8) || reinterpret_cast<const char *>(score) != reinterpret_cast<const char *>(step) + 4;
}

// cudaGetLastError() reports AND clears the thread's sticky launch error, whoever left it there (torch, another library).
// Every entry point therefore discards what was pending before its first launch (clear_stale_error) and checks after
// EACH of its own launches (launch_status), so that a non-zero return always names a launch of this library.
inline void clear_stale_error() { (void)cudaGetLastError(); }

inline int launch_status()
{
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

// Check an n-tuple network given as host arrays (cells [K][6], len [K], stage thresholds stage_exp [S-1]) and expand it into
// the kernels' NTupleStagedSpec: E_NULL (stage_exp only when S > 1), E_SIZE for K, a length or S out of range or a weight
// count other than S * sum 16^len, E_ENUM for a cell > 15, a repeated cell, or thresholds outside 1..15 or not strictly
// ascending
inline int ntuple_spec(const uint8_t *cells, const uint8_t *len, int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages,
                       int64_t num_weights, NTupleStagedSpec &spec)
{
    if (!cells || !len) return ML2048_E_NULL;
    if (num_tuples < 1 || num_tuples > kNTupleMaxTuples) return ML2048_E_SIZE;
    for (int t = 0; t < num_tuples; ++t) {
        if (len[t] < 1 || len[t] > kNTupleMaxLen) return ML2048_E_SIZE;
        uint32_t seen = 0;
        for (int j = 0; j < len[t]; ++j) {
            const uint8_t c = cells[kNTupleMaxLen * t + j];
            if (c > 15 || ((seen >> c) & 1u)) return ML2048_E_ENUM;
            seen |= 1u << c;
        }
    }
    if (num_stages < 1 || num_stages > kNTupleMaxStages) return ML2048_E_SIZE;
    if (num_stages > 1 && !stage_exp) return ML2048_E_NULL;
    for (int k = 0; k + 1 < num_stages; ++k)
        if (stage_exp[k] < 1 || stage_exp[k] > 15 || (k > 0 && stage_exp[k] <= stage_exp[k - 1])) return ML2048_E_ENUM;
    const int64_t n = ntuple_expand(cells, len, num_tuples, spec);
    spec.stage_size = (uint32_t)n;
    spec.stage_of = ntuple_stage_table(stage_exp, num_stages);
    return n * num_stages == num_weights ? 0 : ML2048_E_SIZE;
}

// Runs f(spec) with the spec's single-stage NTupleSpec for a one-stage network (its stage table is all zero: a threshold
// <= 15 puts the board of largest cell 15 in stage >= 1), so S = 1 launches the NTupleSpec instances of the kernels; with
// the staged spec otherwise.  f launches the kernels, templated on the spec type it is given.
template <class F>
inline int with_spec(const NTupleStagedSpec &spec, F &&f)
{
    if (spec.stage_of == 0) return f(static_cast<const NTupleSpec &>(spec));
    return f(spec);
}

// with_spec for the reads and delta phases: a multi-stage network with marks (`promoted` non-null) runs the
// NTuplePromotedSpec instances.  One stage has no mark to read, so it stays the NTupleSpec instances.
template <class F>
inline int with_spec(const NTupleStagedSpec &spec, const uint8_t *promoted, F &&f)
{
    if (!promoted || spec.stage_of == 0) return with_spec(spec, f);
    NTuplePromotedSpec p;
    static_cast<NTupleStagedSpec &>(p) = spec;
    p.promoted = promoted;
    return f(p);
}

// E_NULL / E_ALIGN of the marks of an ml2048_promoted_* entry (4-byte aligned: the promote phase sets them with word atomics)
inline int check_promoted(const uint8_t *promoted)
{
    if (!promoted) return ML2048_E_NULL;
    return misaligned(promoted, 4) ? ML2048_E_ALIGN : 0;
}

constexpr int kMaxDevices = 64;

// index of the current device, or -1 (beyond the per-device tables: callers then take the uncached path)
inline int current_device_slot()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -1;
    return (dev >= 0 && dev < kMaxDevices) ? dev : -1;
}

// Launch as a programmatic dependent of the kernel before it on the stream (the auto-reset scan): see autoreset_scan_kernel.
// ML2048_PDL=0 in the environment keeps the plain stream order (A/B measurements).
inline bool pdl_enabled()
{
    static const bool on = [] { const char *m = getenv("ML2048_PDL"); return !(m && m[0] == '0'); }();
    return on;
}

template <typename... Params, typename... Args>
inline void launch_after_scan(void (*kernel)(Params...), unsigned grid, unsigned block, size_t smem, cudaStream_t s, Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    (void)cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);  // errors surface through launch_status()
}

template <int kRng, bool kLog, bool kFull, bool kReset>
int launch_step_onehot(const ml2048_step_args &a, cudaStream_t s)
{
    // large batches: 768-thread blocks (one contiguous 768 KiB fp32 tile each); medium batches 256-thread blocks; small
    // batches (the training shape) 64-thread blocks, so that the one-hot rows are written by many SMs: M = 2048 is 32
    // blocks instead of 8 (or 3)
    constexpr int T = kOneHotStepThreads;
    constexpr int S = kSmallStepThreads;
    const bool big = a.num_games >= (1 << 19);
    const bool small = a.num_games <= kSmallStepMaxGames;
    const unsigned grid = (unsigned)((a.num_games + kStepThreads - 1) / kStepThreads);
    const unsigned grid_big = (unsigned)((a.num_games + T - 1) / T);
    const unsigned grid_small = (unsigned)((a.num_games + S - 1) / S);
    const int onehot = a.onehot_out ? a.onehot_dtype : ML2048_ONEHOT_NONE;
    if (onehot < ML2048_ONEHOT_NONE || onehot > ML2048_ONEHOT_U8) return ML2048_E_ENUM;
    clear_stale_error();
    // with the auto-reset fused in, the step is a programmatic dependent of the scan that precedes it on the stream
#define ML2048_STEP_LAUNCH(KERNEL, GRID, BLOCK, SMEM)                              \
    do {                                                                           \
        if (kReset) launch_after_scan(KERNEL, GRID, BLOCK, SMEM, s, a);            \
        else KERNEL<<<GRID, BLOCK, SMEM, s>>>(a);                                  \
    } while (0)
#if defined(ML2048_ONEHOT_TMA)
#define ML2048_LAUNCH(OH)                                                                              \
    if (big) {                                                                                         \
        const int smem = kTmaStages * kTmaChunkBytes;                                                  \
        /* > 48 KiB of dynamic shared memory needs an opt-in per kernel AND PER DEVICE (function attributes live in the \
           device's context): one flag per device, like launch_prepare_fused's table */                \
        static bool opted_in[kMaxDevices];                                                             \
        const int dev_slot = current_device_slot();                                                    \
        if (dev_slot < 0 || !opted_in[dev_slot]) {                                                     \
            const cudaError_t e = cudaFuncSetAttribute(step_kernel<kRng, kLog, OH, kFull, T, kReset>,   \
                                                       cudaFuncAttributeMaxDynamicSharedMemorySize, smem); \
            if (e != cudaSuccess) return (int)e;                                                       \
            if (dev_slot >= 0) opted_in[dev_slot] = true;                                              \
        }                                                                                              \
        ML2048_STEP_LAUNCH((step_kernel<kRng, kLog, OH, kFull, T, kReset>), grid_big, T, smem);         \
    } else if (small) ML2048_STEP_LAUNCH((step_kernel<kRng, kLog, OH, kFull, S, kReset>), grid_small, S, 0); \
    else ML2048_STEP_LAUNCH((step_kernel<kRng, kLog, OH, kFull, kStepThreads, kReset>), grid, kStepThreads, 0)
#else
#define ML2048_LAUNCH(OH)                                                                              \
    if (big) ML2048_STEP_LAUNCH((step_kernel<kRng, kLog, OH, kFull, T, kReset>), grid_big, T, 0);       \
    else if (small) ML2048_STEP_LAUNCH((step_kernel<kRng, kLog, OH, kFull, S, kReset>), grid_small, S, 0); \
    else ML2048_STEP_LAUNCH((step_kernel<kRng, kLog, OH, kFull, kStepThreads, kReset>), grid, kStepThreads, 0)
#endif
    switch (onehot) {
    case ML2048_ONEHOT_NONE: ML2048_STEP_LAUNCH((step_kernel<kRng, kLog, ML2048_ONEHOT_NONE, kFull, kStepThreads, kReset>), grid, kStepThreads, 0); break;
    case ML2048_ONEHOT_F32: ML2048_LAUNCH(ML2048_ONEHOT_F32); break;
    case ML2048_ONEHOT_BF16: ML2048_LAUNCH(ML2048_ONEHOT_BF16); break;
    default: ML2048_LAUNCH(ML2048_ONEHOT_U8); break;
    }
#undef ML2048_LAUNCH
#undef ML2048_STEP_LAUNCH
    return launch_status();
}

// A run-time switch of the environment (A/B measurements and tests): whether `on` holds for the value of variable `name`
// (null when unset).  Read once, at first use, or on every call when ML2048_PREPARE_RECHECK was set then (the tests switch
// modes inside one process).  Every caller passes its own lambda and so gets its own instance, with its own cached value.
template <class On>
bool env_switch(const char *name, On on)
{
    static const bool recheck = getenv("ML2048_PREPARE_RECHECK") != nullptr;
    static const bool at_start = on(getenv(name));
    return recheck ? on(getenv(name)) : at_start;
}

// ML2048_STEP=single keeps large lean batches on the one-game-per-thread kernel (the differential test of the two kernels).
inline bool force_single_step()
{
    return env_switch("ML2048_STEP", [](const char *m) { return m && strcmp(m, "single") == 0; });
}

// ML2048_PREPARE=split forces the three-launch auto-reset.
inline bool force_split_prepare()
{
    return env_switch("ML2048_PREPARE", [](const char *m) { return m && m[0] == 's'; });
}

template <int kRng>
int launch_step(const ml2048_step_args &a, cudaStream_t s)
{
    const bool full = a.action_mode == ML2048_ACTIONS_FROM_LOGITS || a.episode_max_tile || a.traj_state || a.tr_state || a.tr_valid_actions ||
                      a.tr_action || a.tr_reward || a.tr_next_state || a.tr_next_valid_actions || a.tr_step || a.tr_terminated;
    const int onehot_kind = a.onehot_out ? a.onehot_dtype : ML2048_ONEHOT_NONE;
    if (!full && !a.merged && onehot_kind == ML2048_ONEHOT_NONE && a.num_games >= kPairMinGames && a.num_games < (1ll << 31) && !force_single_step()) {
        // the lean core-only configuration at large batches: two games per thread
        const unsigned grid = (unsigned)(((a.num_games + 1) / 2 + kPairThreads - 1) / kPairThreads);
        clear_stale_error();
        const bool normal = a.reward_kind == ML2048_REWARD_NORMAL;
        const bool random = a.action_mode == ML2048_ACTIONS_RANDOM_VALID;
        const int variant = (a.reset_rank ? 4 : random ? 2 : 0) + (normal ? 1 : 0);  // the fused auto-reset implies the random policy
        PairConst x;
        x.policy_keys = philox_round_keys(a.philox_seed, 0u);
        x.spawn_keys = philox_round_keys(a.philox_seed, kSpawnStream);
        x.flags = (a.actions_out ? kPairActionsOut : 0u) | (a.stats ? kPairStats : 0u) | (a.age ? kPairAge : 0u) |
                  (a.reset_indices ? kPairResetIndices : 0u) | ((a.slot_base & 1) ? kPairOddSlotBase : 0u) | (a.sched ? kPairSched : 0u);
#define ML2048_PAIR_LAUNCH(RESET, RANDOM, NORMAL)                                                                 \
    if (RESET) launch_after_scan(step_pair_kernel<kRng, RESET, RANDOM, NORMAL>, grid, kPairThreads, 0, s, a, x);  \
    else step_pair_kernel<kRng, RESET, RANDOM, NORMAL><<<grid, kPairThreads, 0, s>>>(a, x)
        switch (variant) {
        case 5: ML2048_PAIR_LAUNCH(true, true, true); break;
        case 4: ML2048_PAIR_LAUNCH(true, true, false); break;
        case 3: ML2048_PAIR_LAUNCH(false, true, true); break;
        case 2: ML2048_PAIR_LAUNCH(false, true, false); break;
        case 1: ML2048_PAIR_LAUNCH(false, false, true); break;
        default: ML2048_PAIR_LAUNCH(false, false, false); break;
        }
#undef ML2048_PAIR_LAUNCH
        return launch_status();
    }
    if (a.reset_rank) {
        // the fused auto-reset is built for the lean kernels (the synthetic random-policy rollouts it serves)
        if (full) return ML2048_E_ENUM;
        return a.merged ? launch_step_onehot<kRng, true, false, true>(a, s) : launch_step_onehot<kRng, false, false, true>(a, s);
    }
    if (full) return a.merged ? launch_step_onehot<kRng, true, true, false>(a, s) : launch_step_onehot<kRng, false, true, false>(a, s);
    return a.merged ? launch_step_onehot<kRng, true, false, false>(a, s) : launch_step_onehot<kRng, false, false, false>(a, s);
}

}  // namespace

// ---- C ABI ----------------------------------------------------------------------------------

extern "C" {

int ml2048_abi_version(void) { return ML2048_ABI_VERSION; }

int64_t ml2048_prepare_scratch_ints(int64_t num_games)
{
    if (num_games <= 0) return 0;
    const int64_t tiles = (num_games + kPrepTile - 1) / kPrepTile;
    return ((tiles + 1) / 2) * 2 + 2;  // tile counts (padded to 8 bytes) + one int64
}

int ml2048_step(const ml2048_step_args *args, void *stream)
{
    if (!args) return ML2048_E_NULL;
    if (args->struct_size != sizeof(ml2048_step_args)) return ML2048_E_STRUCT;
    const ml2048_step_args &a = *args;
    if (a.num_games <= 0) return ML2048_E_SIZE;
    if (!a.board_in || !a.board_out || !a.valid_out || !a.step || !a.score || !a.reward || !a.terminated || !a.invalid)
        return ML2048_E_NULL;
    if (a.board_in == a.board_out) return ML2048_E_NULL;
    if (not_a_step_score_pair(a.step, a.score)) return ML2048_E_ALIGN;
    if (misaligned(a.board_in, 16) || misaligned(a.board_out, 16) || misaligned(a.valid_out, 4) || misaligned(a.merged, 16) ||
        misaligned(a.onehot_out, 16) || misaligned(a.valid_in, 4) || misaligned(a.stats, 8))
        return ML2048_E_ALIGN;
    if (a.reward_kind < 0 || a.reward_kind > ML2048_REWARD_MAXCELL) return ML2048_E_ENUM;
    if (a.action_mode == ML2048_ACTIONS_GIVEN) {
        if (!a.actions) return ML2048_E_NULL;
        if (a.action_dtype < 0 || a.action_dtype > ML2048_ACT_I64) return ML2048_E_ENUM;
        if (misaligned(a.actions, a.action_dtype == ML2048_ACT_I64 ? 8 : (a.action_dtype == ML2048_ACT_I32 ? 4 : 1)))
            return ML2048_E_ALIGN;
    } else if (a.action_mode == ML2048_ACTIONS_RANDOM_VALID) {
        if (!a.valid_in) return ML2048_E_NULL;
    } else if (a.action_mode == ML2048_ACTIONS_FROM_LOGITS) {
        if (!a.valid_in || !a.logits) return ML2048_E_NULL;
        if (misaligned(a.logits, 16) || misaligned(a.log_prob_out, 4)) return ML2048_E_ALIGN;
    } else {
        return ML2048_E_ENUM;
    }
    if (a.tr_valid_actions && !a.valid_in) return ML2048_E_NULL;
    if (misaligned(a.tr_state, 16) || misaligned(a.tr_next_state, 16) || misaligned(a.tr_valid_actions, 4) ||
        misaligned(a.tr_next_valid_actions, 4) || misaligned(a.tr_reward, 4) || misaligned(a.tr_step, 4))
        return ML2048_E_ALIGN;
    if (a.onehot_out && (a.onehot_dtype < ML2048_ONEHOT_F32 || a.onehot_dtype > ML2048_ONEHOT_U8)) return ML2048_E_ENUM;
    if (a.episode_max_tile && (!a.id || !a.episode_steps || !a.episode_score || a.episode_capacity <= 0)) return ML2048_E_NULL;
    if (a.traj_state && (!a.id || !a.age || !a.traj_action || !a.traj_score || !a.traj_rows || a.traj_capacity <= 0 || a.traj_max_rows <= 0))
        return ML2048_E_NULL;
    if (misaligned(a.traj_state, 16) || misaligned(a.traj_score, 4) || misaligned(a.traj_rows, 4) || misaligned(a.age, 4))
        return ML2048_E_ALIGN;
    if (a.sched) {
        if (!a.sched_cursor || a.sched_cursor == a.sched_cursor_next) return ML2048_E_NULL;
        if (misaligned(a.sched, 8) || misaligned(a.sched_cursor, 8) || misaligned(a.sched_cursor_next, 8) || (a.table_stride & 15))
            return ML2048_E_ALIGN;
    }
    if (a.reset_rank) {
        if (a.action_mode != ML2048_ACTIONS_RANDOM_VALID) return ML2048_E_ENUM;  // given actions belong to post-reset observations
        if (!a.reset_chunk_base || !a.reset_id_base || !a.id || !a.valid_in) return ML2048_E_NULL;
        if (a.rng_mode == ML2048_RNG_REPLAY && !a.randperm) return ML2048_E_NULL;
        if (misaligned(a.reset_rank, 4) || misaligned(a.reset_chunk_base, 4) || misaligned(a.reset_id_base, 8) ||
            misaligned(a.reset_indices, 8) || misaligned(a.randperm, 16) || misaligned(a.id, 4))
            return ML2048_E_ALIGN;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (a.rng_mode == ML2048_RNG_REPLAY) {
        if (!a.randperm_keys) return ML2048_E_NULL;
        if (misaligned(a.randperm_keys, 16)) return ML2048_E_ALIGN;
        return launch_step<ML2048_RNG_REPLAY>(a, s);
    }
    if (a.rng_mode == ML2048_RNG_PHILOX) return launch_step<ML2048_RNG_PHILOX>(a, s);
    return ML2048_E_ENUM;
}

static int check_prepare_args(const ml2048_prepare_args *args)
{
    if (!args) return ML2048_E_NULL;
    if (args->struct_size != sizeof(ml2048_prepare_args)) return ML2048_E_STRUCT;
    const ml2048_prepare_args &a = *args;
    if (a.num_games <= 0) return ML2048_E_SIZE;
    if (!a.board || !a.valid || !a.id || !a.step || !a.score || !a.reward || !a.terminated || !a.invalid || !a.game_count ||
        !a.reset_count || !a.scratch)
        return ML2048_E_NULL;
    if (not_a_step_score_pair(a.step, a.score)) return ML2048_E_ALIGN;
    if (misaligned(a.board, 16) || misaligned(a.valid, 4) || misaligned(a.terminated, 16) || misaligned(a.merged, 16) ||
        misaligned(a.onehot, 16) || misaligned(a.randperm, 16) || misaligned(a.scratch, 8) || misaligned(a.game_count, 8) ||
        misaligned(a.reset_count, 8) || misaligned(a.reset_indices, 8) || misaligned(a.id_offset, 8))
        return ML2048_E_ALIGN;
    if (a.onehot && (a.onehot_dtype < ML2048_ONEHOT_F32 || a.onehot_dtype > ML2048_ONEHOT_U8)) return ML2048_E_ENUM;
    if (a.rng_mode == ML2048_RNG_REPLAY && !a.randperm) return ML2048_E_NULL;
    if (a.rng_mode != ML2048_RNG_REPLAY && a.rng_mode != ML2048_RNG_PHILOX) return ML2048_E_ENUM;
    if (a.sched) {
        if (!a.sched_cursor) return ML2048_E_NULL;
        if (misaligned(a.sched, 8) || misaligned(a.sched_cursor, 8) || (a.table_stride & 15)) return ML2048_E_ALIGN;
    }
    return 0;
}

static inline int64_t *prepare_id_base_slot(const ml2048_prepare_args &a, int tiles)
{
    return reinterpret_cast<int64_t *>(a.scratch + ((tiles + 1) / 2) * 2);
}

int ml2048_prepare_count(const ml2048_prepare_args *args, void *stream)
{
    const int rc = check_prepare_args(args);
    if (rc) return rc;
    const ml2048_prepare_args &a = *args;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t n16 = (a.num_games + 15) / 16;
    const int tiles = (int)((a.num_games + kPrepTile - 1) / kPrepTile);
    clear_stale_error();
    prepare_count_kernel<<<tiles, kPrepThreads, 0, s>>>(reinterpret_cast<const uint4 *>(a.terminated), n16, a.scratch);
    if (const int rc_count = launch_status()) return rc_count;
    prepare_scan_kernel<<<1, kPrepScanThreads, 0, s>>>(a.scratch, tiles, prepare_id_base_slot(a, tiles), a.game_count,
                                                       a.id_offset ? 0 : 1, a.reset_count);
    return launch_status();
}

int ml2048_prepare_apply(const ml2048_prepare_args *args, void *stream)
{
    const int rc = check_prepare_args(args);
    if (rc) return rc;
    const ml2048_prepare_args &a = *args;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int tiles = (int)((a.num_games + kPrepTile - 1) / kPrepTile);
    clear_stale_error();
    if (a.rng_mode == ML2048_RNG_REPLAY)
        prepare_apply_kernel<ML2048_RNG_REPLAY><<<tiles, kPrepThreads, 0, s>>>(a, a.scratch, prepare_id_base_slot(a, tiles));
    else
        prepare_apply_kernel<ML2048_RNG_PHILOX><<<tiles, kPrepThreads, 0, s>>>(a, a.scratch, prepare_id_base_slot(a, tiles));
    return launch_status();
}

// Single-wave cooperative launch of the fused auto-reset; ML2048_E_SIZE when the batch (or the device) does not allow it.
static int launch_prepare_fused(const ml2048_prepare_args &a, cudaStream_t s)
{
    static int max_blocks[kMaxDevices][2];  // co-resident blocks per device and rng mode; 0 = not asked yet, -1 = unavailable
    const int mode = a.rng_mode == ML2048_RNG_REPLAY ? 0 : 1;
    const void *kernel = mode == 0 ? (const void *)prepare_fused_kernel<ML2048_RNG_REPLAY> : (const void *)prepare_fused_kernel<ML2048_RNG_PHILOX>;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    if (dev < 0 || dev >= kMaxDevices) return ML2048_E_SIZE;
    int &blocks_here = max_blocks[dev][mode];
    if (blocks_here == 0) {
        int sms = 0, per_sm = 0, coop = 0;
        e = cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kPrepThreads, 0);
        if (e != cudaSuccess) return (int)e;
        blocks_here = coop && sms * per_sm > 0 ? sms * per_sm : -1;
    }
    if (blocks_here <= 0) return ML2048_E_SIZE;
    const int64_t n16 = (a.num_games + 15) / 16;
    const int64_t tiles = (a.num_games + kPrepTile - 1) / kPrepTile;  // the scratch holds one int per tile
    const int64_t blocks = tiles < blocks_here ? tiles : blocks_here;
    if ((n16 + blocks - 1) / blocks > kFusedMaxGroups) return ML2048_E_SIZE;
    clear_stale_error();
    ml2048_prepare_args args = a;
    int32_t *counts = a.scratch;
    void *params[] = {&args, &counts};
    e = cudaLaunchCooperativeKernel(kernel, dim3((unsigned)blocks), dim3(kPrepThreads), params, 0, s);
    if (e == cudaErrorCooperativeLaunchTooLarge) {
        // fewer SMs are available to this context than the device reports (MPS share, green context): three launches
        (void)cudaGetLastError();
        blocks_here = -1;
        return ML2048_E_SIZE;
    }
    return e == cudaSuccess ? launch_status() : (int)e;
}

int ml2048_prepare(const ml2048_prepare_args *args, void *stream)
{
    int rc = check_prepare_args(args);
    if (rc) return rc;
    if (args->num_games <= kPrepSmallMaxGames && !args->id_offset) {
        cudaStream_t s = static_cast<cudaStream_t>(stream);
        clear_stale_error();
        if (args->rng_mode == ML2048_RNG_REPLAY)
            prepare_small_kernel<ML2048_RNG_REPLAY><<<1, kPrepThreads, 0, s>>>(*args);
        else
            prepare_small_kernel<ML2048_RNG_PHILOX><<<1, kPrepThreads, 0, s>>>(*args);
        return launch_status();
    }
    if (!args->id_offset && !force_split_prepare()) {
        rc = launch_prepare_fused(*args, static_cast<cudaStream_t>(stream));
        if (rc != ML2048_E_SIZE) return rc;  // E_SIZE: the batch does not fit the single-wave kernel, use three launches
    }
    rc = ml2048_prepare_count(args, stream);
    if (rc) return rc;
    return ml2048_prepare_apply(args, stream);
}

int64_t ml2048_autoreset_scratch_ints(int64_t num_games)
{
    if (num_games <= 0) return 0;
    const int64_t groups = (num_games + 31) / 32;
    return (groups + kScanThreads - 1) / kScanThreads + 2;
}

int ml2048_autoreset_scan(const uint8_t *terminated, int32_t *reset_rank, int32_t *reset_chunk_base, int64_t num_games, int64_t *game_count,
                          const int64_t *id_offset, int64_t *reset_id_base, int64_t *reset_count, int32_t *scratch, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!terminated || !reset_rank || !reset_chunk_base || !game_count || !reset_id_base || !reset_count || !scratch) return ML2048_E_NULL;
    if (misaligned(terminated, 16) || misaligned(reset_rank, 4) || misaligned(reset_chunk_base, 4) || misaligned(game_count, 8) ||
        misaligned(id_offset, 8) || misaligned(reset_id_base, 8) || misaligned(reset_count, 8) || misaligned(scratch, 4))
        return ML2048_E_ALIGN;
    const int64_t groups = (num_games + 31) / 32;
    const unsigned chunks = (unsigned)((groups + kScanThreads - 1) / kScanThreads);
    clear_stale_error();
    autoreset_scan_kernel<<<chunks, kScanThreads, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const uint4 *>(terminated),
                                                                                        (num_games + 15) / 16, reset_rank, reset_chunk_base, groups,
                                                                                        game_count, id_offset, reset_id_base, reset_count,
                                                                                        scratch);
    return launch_status();
}

int ml2048_reset_state(void *board_a, void *board_b, void *valid_a, void *valid_b, int32_t *id, int32_t *step, float *score,
                       float *reward, uint8_t *terminated, uint8_t *invalid, uint8_t *merged, int64_t num_games, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!board_a || !board_b || !valid_a || !valid_b || !id || !step || !score || !reward || !terminated || !invalid)
        return ML2048_E_NULL;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t n = (size_t)num_games;
    if (not_a_step_score_pair(step, score)) return ML2048_E_ALIGN;
    const struct { void *p; size_t bytes; } clears[] = {{board_a, n * 16}, {board_b, n * 16}, {valid_a, n * 4}, {valid_b, n * 4},
                                                        {id, n * 4},       {step, n * 8} /* {step, score} pairs */, {reward, n * 4},
                                                        {invalid, n},      {merged, n * 16}};
    for (const auto &c : clears) {
        if (!c.p) continue;
        const cudaError_t e = cudaMemsetAsync(c.p, 0, c.bytes, s);
        if (e != cudaSuccess) return (int)e;
    }
    const int64_t padded = (num_games + 15) / 16 * 16;
    clear_stale_error();
    fill_terminated_kernel<<<(unsigned)((padded + 255) / 256), 256, 0, s>>>(terminated, num_games, padded);
    return launch_status();
}

int ml2048_encode_onehot(const void *board, void *out, int32_t onehot_dtype, int64_t num_games, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!board || !out) return ML2048_E_NULL;
    if (misaligned(board, 16) || misaligned(out, 16)) return ML2048_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const unsigned grid = (unsigned)((num_games + kStepThreads - 1) / kStepThreads);
    const uint4 *b = reinterpret_cast<const uint4 *>(board);
    clear_stale_error();
    switch (onehot_dtype) {
    case ML2048_ONEHOT_F32: onehot_kernel<ML2048_ONEHOT_F32><<<grid, kStepThreads, 0, s>>>(b, out, num_games); break;
    case ML2048_ONEHOT_BF16: onehot_kernel<ML2048_ONEHOT_BF16><<<grid, kStepThreads, 0, s>>>(b, out, num_games); break;
    case ML2048_ONEHOT_U8: onehot_kernel<ML2048_ONEHOT_U8><<<grid, kStepThreads, 0, s>>>(b, out, num_games); break;
    default: return ML2048_E_ENUM;
    }
    return launch_status();
}

int ml2048_valid_actions(const void *board, void *valid_out, int64_t num_games, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!board || !valid_out) return ML2048_E_NULL;
    if (misaligned(board, 16) || misaligned(valid_out, 4)) return ML2048_E_ALIGN;
    const unsigned grid = (unsigned)((num_games + kStepThreads - 1) / kStepThreads);
    clear_stale_error();
    valid_kernel<<<grid, kStepThreads, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const uint4 *>(board),
                                                                                reinterpret_cast<uint32_t *>(valid_out), num_games);
    return launch_status();
}

int ml2048_afterstates(const void *board, void *after_out, float *reward_out, uint8_t *valid_out, uint8_t *merged_out, int32_t reward_kind,
                       int64_t num_games, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!board || !after_out || !reward_out || !valid_out) return ML2048_E_NULL;
    if (misaligned(board, 16) || misaligned(after_out, 16) || misaligned(merged_out, 16) || misaligned(reward_out, 4)) return ML2048_E_ALIGN;
    if (reward_kind < 0 || reward_kind > ML2048_REWARD_MAXCELL) return ML2048_E_ENUM;
    const int64_t grid = (num_games + kStepThreads / 4 - 1) / (kStepThreads / 4);  // four threads per game
    if (grid > 0x7fffffff) return ML2048_E_SIZE;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const uint4 *b = reinterpret_cast<const uint4 *>(board);
    uint4 *after = reinterpret_cast<uint4 *>(after_out), *merged = reinterpret_cast<uint4 *>(merged_out);
    clear_stale_error();
    if (merged)
        afterstates_kernel<true><<<(unsigned)grid, kStepThreads, 0, s>>>(b, after, reward_out, valid_out, merged, reward_kind, num_games);
    else
        afterstates_kernel<false><<<(unsigned)grid, kStepThreads, 0, s>>>(b, after, reward_out, valid_out, merged, reward_kind, num_games);
    return launch_status();
}

static int value_entry(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                       int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages, const uint8_t *promoted, float *value_out,
                       int64_t num_games, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!board || !weights || !value_out) return ML2048_E_NULL;
    if (misaligned(board, 16) || misaligned(weights, 4) || misaligned(value_out, 4)) return ML2048_E_ALIGN;
    NTupleStagedSpec spec;
    if (const int rc = ntuple_spec(cells, len, num_tuples, stage_exp, num_stages, num_weights, spec)) return rc;
    const int64_t grid = (num_games + kStepThreads - 1) / kStepThreads;
    if (grid > 0x7fffffff) return ML2048_E_SIZE;
    clear_stale_error();
    return with_spec(spec, promoted, [&](const auto &sp) {
        ntuple_value_kernel<<<(unsigned)grid, kStepThreads, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const uint4 *>(board),
                                                                                                 weights, sp, value_out, num_games);
        return launch_status();
    });
}

int ml2048_staged_value(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                        int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages, float *value_out, int64_t num_games,
                        void *stream)
{
    return value_entry(board, weights, num_weights, cells, len, num_tuples, stage_exp, num_stages, nullptr, value_out, num_games, stream);
}

int ml2048_promoted_value(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                          int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages, const uint8_t *promoted, float *value_out,
                          int64_t num_games, void *stream)
{
    if (const int rc = check_promoted(promoted)) return rc;
    return value_entry(board, weights, num_weights, cells, len, num_tuples, stage_exp, num_stages, promoted, value_out, num_games, stream);
}

int ml2048_ntuple_value(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                        int32_t num_tuples, float *value_out, int64_t num_games, void *stream)
{
    return ml2048_staged_value(board, weights, num_weights, cells, len, num_tuples, nullptr, 1, value_out, num_games, stream);
}

static int greedy_entry(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                        int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages, const uint8_t *promoted, int32_t reward_kind,
                        uint8_t *action_u8, int64_t *action_i64, void *after_out, float *reward_out, float *value_out, int64_t num_games,
                        void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!board || !weights || (!action_u8 && !action_i64) || !after_out || !reward_out || !value_out) return ML2048_E_NULL;
    if (misaligned(board, 16) || misaligned(weights, 4) || misaligned(action_i64, 8) || misaligned(after_out, 16) ||
        misaligned(reward_out, 4) || misaligned(value_out, 4))
        return ML2048_E_ALIGN;
    if (reward_kind < 0 || reward_kind > ML2048_REWARD_MAXCELL) return ML2048_E_ENUM;
    NTupleStagedSpec spec;
    if (const int rc = ntuple_spec(cells, len, num_tuples, stage_exp, num_stages, num_weights, spec)) return rc;
    const int64_t grid = (num_games + kStepThreads / 4 - 1) / (kStepThreads / 4);  // four threads per game
    if (grid > 0x7fffffff) return ML2048_E_SIZE;
    clear_stale_error();
    return with_spec(spec, promoted, [&](const auto &sp) {
        ntuple_greedy_kernel<<<(unsigned)grid, kStepThreads, 0, static_cast<cudaStream_t>(stream)>>>(
            reinterpret_cast<const uint4 *>(board), weights, sp, reward_kind, action_u8, reinterpret_cast<long long *>(action_i64),
            reinterpret_cast<uint4 *>(after_out), reward_out, value_out, num_games);
        return launch_status();
    });
}

int ml2048_staged_greedy(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                         int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages, int32_t reward_kind, uint8_t *action_u8,
                         int64_t *action_i64, void *after_out, float *reward_out, float *value_out, int64_t num_games, void *stream)
{
    return greedy_entry(board, weights, num_weights, cells, len, num_tuples, stage_exp, num_stages, nullptr, reward_kind, action_u8,
                        action_i64, after_out, reward_out, value_out, num_games, stream);
}

int ml2048_promoted_greedy(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                           int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages, const uint8_t *promoted, int32_t reward_kind,
                           uint8_t *action_u8, int64_t *action_i64, void *after_out, float *reward_out, float *value_out,
                           int64_t num_games, void *stream)
{
    if (const int rc = check_promoted(promoted)) return rc;
    return greedy_entry(board, weights, num_weights, cells, len, num_tuples, stage_exp, num_stages, promoted, reward_kind, action_u8,
                        action_i64, after_out, reward_out, value_out, num_games, stream);
}

int ml2048_ntuple_greedy(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                         int32_t num_tuples, int32_t reward_kind, uint8_t *action_u8, int64_t *action_i64, void *after_out,
                         float *reward_out, float *value_out, int64_t num_games, void *stream)
{
    return ml2048_staged_greedy(board, weights, num_weights, cells, len, num_tuples, nullptr, 1, reward_kind, action_u8, action_i64,
                                after_out, reward_out, value_out, num_games, stream);
}

static int expectimax_entry(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                            int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages, const uint8_t *promoted,
                            int32_t reward_kind, int32_t depth, double two_prob, uint8_t *action_u8, int64_t *action_i64,
                            void *after_out, float *reward_out, float *value_out, float *q_out, int64_t num_games, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!board || !weights || (!action_u8 && !action_i64) || !after_out || !reward_out || !value_out || !q_out) return ML2048_E_NULL;
    if (misaligned(board, 16) || misaligned(weights, 4) || misaligned(action_i64, 8) || misaligned(after_out, 16) ||
        misaligned(reward_out, 4) || misaligned(value_out, 4) || misaligned(q_out, 4))
        return ML2048_E_ALIGN;
    if (reward_kind < 0 || reward_kind > ML2048_REWARD_MAXCELL || (depth != 1 && depth != 2) || !(two_prob >= 0.0 && two_prob <= 1.0))
        return ML2048_E_ENUM;
    NTupleStagedSpec spec;
    if (const int rc = ntuple_spec(cells, len, num_tuples, stage_exp, num_stages, num_weights, spec)) return rc;
    SpawnLaw law;
    law.p2 = (float)two_prob;
    law.p4 = 1.0f - law.p2;
    const int64_t per_block = depth == 1 ? kExpectimax1BoardsPerBlock : 1;
    const int64_t grid = (num_games + per_block - 1) / per_block;
    if (grid > 0x7fffffff) return ML2048_E_SIZE;
    const uint4 *b = reinterpret_cast<const uint4 *>(board);
    long long *a64 = reinterpret_cast<long long *>(action_i64);
    uint4 *after = reinterpret_cast<uint4 *>(after_out);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    clear_stale_error();
    return with_spec(spec, promoted, [&](const auto &sp) {
        if (depth == 1)
            expectimax1_kernel<<<(unsigned)grid, kExpectimaxThreads, 0, s>>>(b, weights, sp, reward_kind, law, action_u8, a64, after,
                                                                             reward_out, value_out, q_out, num_games);
        else
            expectimax2_kernel<<<(unsigned)grid, kExpectimaxThreads, 0, s>>>(b, weights, sp, reward_kind, law, action_u8, a64, after,
                                                                             reward_out, value_out, q_out);
        return launch_status();
    });
}

int ml2048_staged_expectimax(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                             int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages, int32_t reward_kind, int32_t depth,
                             double two_prob, uint8_t *action_u8, int64_t *action_i64, void *after_out, float *reward_out,
                             float *value_out, float *q_out, int64_t num_games, void *stream)
{
    return expectimax_entry(board, weights, num_weights, cells, len, num_tuples, stage_exp, num_stages, nullptr, reward_kind, depth,
                            two_prob, action_u8, action_i64, after_out, reward_out, value_out, q_out, num_games, stream);
}

int ml2048_promoted_expectimax(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                               int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages, const uint8_t *promoted,
                               int32_t reward_kind, int32_t depth, double two_prob, uint8_t *action_u8, int64_t *action_i64,
                               void *after_out, float *reward_out, float *value_out, float *q_out, int64_t num_games, void *stream)
{
    if (const int rc = check_promoted(promoted)) return rc;
    return expectimax_entry(board, weights, num_weights, cells, len, num_tuples, stage_exp, num_stages, promoted, reward_kind, depth,
                            two_prob, action_u8, action_i64, after_out, reward_out, value_out, q_out, num_games, stream);
}

int ml2048_expectimax(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples,
                      int32_t reward_kind, int32_t depth, double two_prob, uint8_t *action_u8, int64_t *action_i64, void *after_out,
                      float *reward_out, float *value_out, float *q_out, int64_t num_games, void *stream)
{
    return ml2048_staged_expectimax(board, weights, num_weights, cells, len, num_tuples, nullptr, 1, reward_kind, depth, two_prob, action_u8,
                                    action_i64, after_out, reward_out, value_out, q_out, num_games, stream);
}

// Checks every n-tuple update shares: the batch, the afterstates (x_0's, or the ring that holds them), the float32 values the
// delta starts from (the target, or the reward ring), the weights, the delta output and the network with its stages.  On
// success `spec` and `grid` (one thread per game) are ready for the launches.
static int check_update(const void *after, const float *values, const float *weights, const float *delta_out, int64_t num_weights,
                        const uint8_t *cells, const uint8_t *len, int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages,
                        int64_t num_games, NTupleStagedSpec &spec, unsigned &grid)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!after || !values || !weights || !delta_out) return ML2048_E_NULL;
    if (misaligned(after, 16) || misaligned(values, 4) || misaligned(weights, 4) || misaligned(delta_out, 4)) return ML2048_E_ALIGN;
    if (const int rc = ntuple_spec(cells, len, num_tuples, stage_exp, num_stages, num_weights, spec)) return rc;
    const int64_t blocks = (num_games + kStepThreads - 1) / kStepThreads;
    if (blocks > 0x7fffffff) return ML2048_E_SIZE;
    grid = (unsigned)blocks;
    return 0;
}

// Phase 1 of TD(0) and TC: delta = alpha * (target - V(after))
static int target_delta(const uint4 *after, const float *target, const uint8_t *mask, float alpha, const float *weights,
                        const NTupleStagedSpec &spec, const uint8_t *promoted, float *delta_out, unsigned grid, int64_t num_games,
                        cudaStream_t s)
{
    clear_stale_error();
    return with_spec(spec, promoted, [&](const auto &sp) {
        ntuple_td_delta_kernel<<<grid, kStepThreads, 0, s>>>(after, target, mask, alpha, weights, sp, delta_out, num_games);
        return launch_status();
    });
}

// Phase 1 of TD(lambda) and TC(lambda): the checks only they make, then delta over the ring.  `x0` = x_0's slot of the ring.
static int lambda_delta(const uint4 *ring, const float *reward_ring, const uint8_t *ended_ring, int32_t horizon, int32_t newest,
                        float lambda, const uint8_t *mask, float alpha, const float *weights, const NTupleStagedSpec &spec,
                        const uint8_t *promoted, float *delta_out, unsigned grid, int64_t num_games, cudaStream_t s, const uint4 *&x0)
{
    if (!ended_ring) return ML2048_E_NULL;
    if (horizon < 1 || horizon > kLambdaMaxHorizon || newest < 0 || newest > horizon) return ML2048_E_SIZE;
    if (!(lambda >= 0.0f && lambda <= 1.0f)) return ML2048_E_ENUM;  // NaN fails both
    x0 = ring + (int64_t)(newest == horizon ? 0 : newest + 1) * num_games;
    const float c = 1.0f - lambda;
    clear_stale_error();
    return with_spec(spec, promoted, [&](const auto &sp) {
        ntuple_lambda_delta_kernel<<<grid, kStepThreads, 0, s>>>(ring, reward_ring, ended_ring, mask, horizon, newest, lambda, c, alpha,
                                                                 weights, sp, delta_out, num_games);
        return launch_status();
    });
}

// The update of x_0's entries after phase 1, on the same stream (so every delta is computed before any weight is written):
// with marks (`promoted` non-null) and S > 1 first the promote phase, then TD(0)'s scatter when `coherence` is null, else
// TC's phases 2 and 3.  The entries are those of x_0's stage.
static int apply_update(const uint4 *x0, const uint8_t *mask, const float *delta, float *weights, float *coherence, float *accum,
                        const NTupleStagedSpec &spec, uint8_t *promoted, unsigned grid, int64_t num_games, cudaStream_t s)
{
    if (promoted && spec.stage_of != 0) {
        ntuple_promote_kernel<<<grid, kStepThreads, 0, s>>>(x0, mask, weights, reinterpret_cast<float2 *>(coherence),
                                                            reinterpret_cast<uint32_t *>(promoted), spec, num_games);
        if (const int rc = launch_status()) return rc;
    }
    return with_spec(spec, [&](const auto &sp) {
        if (!coherence) {
            ntuple_td_scatter_kernel<<<grid, kStepThreads, 0, s>>>(x0, mask, delta, weights, sp, num_games);
            return launch_status();
        }
        ntuple_tc_accumulate_kernel<<<grid, kStepThreads, 0, s>>>(x0, mask, delta, reinterpret_cast<float2 *>(accum), sp, num_games);
        if (const int rc = launch_status()) return rc;
        ntuple_tc_apply_kernel<<<grid, kStepThreads, 0, s>>>(x0, mask, weights, reinterpret_cast<float2 *>(coherence),
                                                             reinterpret_cast<unsigned long long *>(accum), sp, num_games);
        return launch_status();
    });
}

static int td_update_entry(const void *after, const float *target, const uint8_t *mask, float alpha, float *weights, int64_t num_weights,
                           const uint8_t *cells, const uint8_t *len, int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages,
                           uint8_t *promoted, float *delta_out, int64_t num_games, void *stream)
{
    NTupleStagedSpec spec;
    unsigned grid = 0;
    if (const int rc = check_update(after, target, weights, delta_out, num_weights, cells, len, num_tuples, stage_exp, num_stages, num_games,
                                    spec, grid))
        return rc;
    const uint4 *b = reinterpret_cast<const uint4 *>(after);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (const int rc = target_delta(b, target, mask, alpha, weights, spec, promoted, delta_out, grid, num_games, s)) return rc;
    return apply_update(b, mask, delta_out, weights, nullptr, nullptr, spec, promoted, grid, num_games, s);
}

int ml2048_staged_td_update(const void *after, const float *target, const uint8_t *mask, float alpha, float *weights, int64_t num_weights,
                            const uint8_t *cells, const uint8_t *len, int32_t num_tuples, const uint8_t *stage_exp, int32_t num_stages,
                            float *delta_out, int64_t num_games, void *stream)
{
    return td_update_entry(after, target, mask, alpha, weights, num_weights, cells, len, num_tuples, stage_exp, num_stages, nullptr,
                           delta_out, num_games, stream);
}

int ml2048_promoted_td_update(const void *after, const float *target, const uint8_t *mask, float alpha, float *weights,
                              int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples, const uint8_t *stage_exp,
                              int32_t num_stages, uint8_t *promoted, float *delta_out, int64_t num_games, void *stream)
{
    if (const int rc = check_promoted(promoted)) return rc;
    return td_update_entry(after, target, mask, alpha, weights, num_weights, cells, len, num_tuples, stage_exp, num_stages, promoted,
                           delta_out, num_games, stream);
}

int ml2048_ntuple_td_update(const void *after, const float *target, const uint8_t *mask, float alpha, float *weights, int64_t num_weights,
                            const uint8_t *cells, const uint8_t *len, int32_t num_tuples, float *delta_out, int64_t num_games, void *stream)
{
    return ml2048_staged_td_update(after, target, mask, alpha, weights, num_weights, cells, len, num_tuples, nullptr, 1, delta_out, num_games,
                                   stream);
}

static int tc_update_entry(const void *after, const float *target, const uint8_t *mask, float alpha, float *weights, float *coherence,
                           float *accum, int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples,
                           const uint8_t *stage_exp, int32_t num_stages, uint8_t *promoted, float *delta_out, int64_t num_games,
                           void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!coherence || !accum) return ML2048_E_NULL;
    if (misaligned(coherence, 8) || misaligned(accum, 8)) return ML2048_E_ALIGN;
    NTupleStagedSpec spec;
    unsigned grid = 0;
    if (const int rc = check_update(after, target, weights, delta_out, num_weights, cells, len, num_tuples, stage_exp, num_stages, num_games,
                                    spec, grid))
        return rc;
    const uint4 *b = reinterpret_cast<const uint4 *>(after);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (const int rc = target_delta(b, target, mask, alpha, weights, spec, promoted, delta_out, grid, num_games, s)) return rc;
    return apply_update(b, mask, delta_out, weights, coherence, accum, spec, promoted, grid, num_games, s);
}

int ml2048_staged_tc_update(const void *after, const float *target, const uint8_t *mask, float alpha, float *weights, float *coherence,
                            float *accum, int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples,
                            const uint8_t *stage_exp, int32_t num_stages, float *delta_out, int64_t num_games, void *stream)
{
    return tc_update_entry(after, target, mask, alpha, weights, coherence, accum, num_weights, cells, len, num_tuples, stage_exp, num_stages,
                           nullptr, delta_out, num_games, stream);
}

int ml2048_promoted_tc_update(const void *after, const float *target, const uint8_t *mask, float alpha, float *weights, float *coherence,
                              float *accum, int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples,
                              const uint8_t *stage_exp, int32_t num_stages, uint8_t *promoted, float *delta_out, int64_t num_games,
                              void *stream)
{
    if (const int rc = check_promoted(promoted)) return rc;
    return tc_update_entry(after, target, mask, alpha, weights, coherence, accum, num_weights, cells, len, num_tuples, stage_exp, num_stages,
                           promoted, delta_out, num_games, stream);
}

int ml2048_tc_update(const void *after, const float *target, const uint8_t *mask, float alpha, float *weights, float *coherence,
                     float *accum, int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples, float *delta_out,
                     int64_t num_games, void *stream)
{
    return ml2048_staged_tc_update(after, target, mask, alpha, weights, coherence, accum, num_weights, cells, len, num_tuples, nullptr, 1,
                                   delta_out, num_games, stream);
}

static int lambda_td_update_entry(const void *after_ring, const float *reward_ring, const uint8_t *ended_ring, int32_t horizon,
                                  int32_t newest, float lambda, const uint8_t *mask, float alpha, float *weights, int64_t num_weights,
                                  const uint8_t *cells, const uint8_t *len, int32_t num_tuples, const uint8_t *stage_exp,
                                  int32_t num_stages, uint8_t *promoted, float *delta_out, int64_t num_games, void *stream)
{
    NTupleStagedSpec spec;
    unsigned grid = 0;
    if (const int rc = check_update(after_ring, reward_ring, weights, delta_out, num_weights, cells, len, num_tuples, stage_exp, num_stages,
                                    num_games, spec, grid))
        return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const uint4 *x0 = nullptr;
    if (const int rc = lambda_delta(reinterpret_cast<const uint4 *>(after_ring), reward_ring, ended_ring, horizon, newest, lambda, mask, alpha,
                                    weights, spec, promoted, delta_out, grid, num_games, s, x0))
        return rc;
    return apply_update(x0, mask, delta_out, weights, nullptr, nullptr, spec, promoted, grid, num_games, s);
}

int ml2048_staged_lambda_td_update(const void *after_ring, const float *reward_ring, const uint8_t *ended_ring, int32_t horizon,
                                   int32_t newest, float lambda, const uint8_t *mask, float alpha, float *weights, int64_t num_weights,
                                   const uint8_t *cells, const uint8_t *len, int32_t num_tuples, const uint8_t *stage_exp,
                                   int32_t num_stages, float *delta_out, int64_t num_games, void *stream)
{
    return lambda_td_update_entry(after_ring, reward_ring, ended_ring, horizon, newest, lambda, mask, alpha, weights, num_weights, cells, len,
                                  num_tuples, stage_exp, num_stages, nullptr, delta_out, num_games, stream);
}

int ml2048_promoted_lambda_td_update(const void *after_ring, const float *reward_ring, const uint8_t *ended_ring, int32_t horizon,
                                     int32_t newest, float lambda, const uint8_t *mask, float alpha, float *weights, int64_t num_weights,
                                     const uint8_t *cells, const uint8_t *len, int32_t num_tuples, const uint8_t *stage_exp,
                                     int32_t num_stages, uint8_t *promoted, float *delta_out, int64_t num_games, void *stream)
{
    if (const int rc = check_promoted(promoted)) return rc;
    return lambda_td_update_entry(after_ring, reward_ring, ended_ring, horizon, newest, lambda, mask, alpha, weights, num_weights, cells, len,
                                  num_tuples, stage_exp, num_stages, promoted, delta_out, num_games, stream);
}

int ml2048_lambda_td_update(const void *after_ring, const float *reward_ring, const uint8_t *ended_ring, int32_t horizon, int32_t newest,
                            float lambda, const uint8_t *mask, float alpha, float *weights, int64_t num_weights, const uint8_t *cells,
                            const uint8_t *len, int32_t num_tuples, float *delta_out, int64_t num_games, void *stream)
{
    return ml2048_staged_lambda_td_update(after_ring, reward_ring, ended_ring, horizon, newest, lambda, mask, alpha, weights, num_weights,
                                          cells, len, num_tuples, nullptr, 1, delta_out, num_games, stream);
}

static int lambda_tc_update_entry(const void *after_ring, const float *reward_ring, const uint8_t *ended_ring, int32_t horizon,
                                  int32_t newest, float lambda, const uint8_t *mask, float alpha, float *weights, float *coherence,
                                  float *accum, int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples,
                                  const uint8_t *stage_exp, int32_t num_stages, uint8_t *promoted, float *delta_out, int64_t num_games,
                                  void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!coherence || !accum) return ML2048_E_NULL;
    if (misaligned(coherence, 8) || misaligned(accum, 8)) return ML2048_E_ALIGN;
    NTupleStagedSpec spec;
    unsigned grid = 0;
    if (const int rc = check_update(after_ring, reward_ring, weights, delta_out, num_weights, cells, len, num_tuples, stage_exp, num_stages,
                                    num_games, spec, grid))
        return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const uint4 *x0 = nullptr;
    if (const int rc = lambda_delta(reinterpret_cast<const uint4 *>(after_ring), reward_ring, ended_ring, horizon, newest, lambda, mask, alpha,
                                    weights, spec, promoted, delta_out, grid, num_games, s, x0))
        return rc;
    return apply_update(x0, mask, delta_out, weights, coherence, accum, spec, promoted, grid, num_games, s);
}

int ml2048_staged_lambda_tc_update(const void *after_ring, const float *reward_ring, const uint8_t *ended_ring, int32_t horizon,
                                   int32_t newest, float lambda, const uint8_t *mask, float alpha, float *weights, float *coherence,
                                   float *accum, int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples,
                                   const uint8_t *stage_exp, int32_t num_stages, float *delta_out, int64_t num_games, void *stream)
{
    return lambda_tc_update_entry(after_ring, reward_ring, ended_ring, horizon, newest, lambda, mask, alpha, weights, coherence, accum,
                                  num_weights, cells, len, num_tuples, stage_exp, num_stages, nullptr, delta_out, num_games, stream);
}

int ml2048_promoted_lambda_tc_update(const void *after_ring, const float *reward_ring, const uint8_t *ended_ring, int32_t horizon,
                                     int32_t newest, float lambda, const uint8_t *mask, float alpha, float *weights, float *coherence,
                                     float *accum, int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples,
                                     const uint8_t *stage_exp, int32_t num_stages, uint8_t *promoted, float *delta_out,
                                     int64_t num_games, void *stream)
{
    if (const int rc = check_promoted(promoted)) return rc;
    return lambda_tc_update_entry(after_ring, reward_ring, ended_ring, horizon, newest, lambda, mask, alpha, weights, coherence, accum,
                                  num_weights, cells, len, num_tuples, stage_exp, num_stages, promoted, delta_out, num_games, stream);
}

int ml2048_lambda_tc_update(const void *after_ring, const float *reward_ring, const uint8_t *ended_ring, int32_t horizon, int32_t newest,
                            float lambda, const uint8_t *mask, float alpha, float *weights, float *coherence, float *accum,
                            int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples, float *delta_out,
                            int64_t num_games, void *stream)
{
    return ml2048_staged_lambda_tc_update(after_ring, reward_ring, ended_ring, horizon, newest, lambda, mask, alpha, weights, coherence, accum,
                                          num_weights, cells, len, num_tuples, nullptr, 1, delta_out, num_games, stream);
}

int ml2048_pack_flags(const void *valid, const uint8_t *terminated, const uint8_t *invalid, uint8_t *packed, int64_t num_games, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!valid || !packed) return ML2048_E_NULL;
    if (misaligned(valid, 4)) return ML2048_E_ALIGN;
    const unsigned grid = (unsigned)(((num_games + 3) / 4 + kStepThreads - 1) / kStepThreads);
    clear_stale_error();
    pack_flags_kernel<<<grid, kStepThreads, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const uint32_t *>(valid), terminated, invalid,
                                                                                  packed, num_games);
    return launch_status();
}

int ml2048_max_tile_hist(const void *board, const uint8_t *terminated, int64_t num_games, unsigned long long *hist20, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!board || !hist20) return ML2048_E_NULL;
    if (misaligned(board, 16) || misaligned(hist20, 8)) return ML2048_E_ALIGN;
    int64_t grid = (num_games + kStepThreads - 1) / kStepThreads;
    if (grid > 148 * 8) grid = 148 * 8;
    clear_stale_error();
    max_tile_hist_kernel<<<(unsigned)grid, kStepThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const uint4 *>(board), terminated, num_games, hist20);
    return launch_status();
}

int ml2048_sample_random_valid(const void *valid, uint8_t *actions_out, int64_t num_games, int64_t slot_base, uint64_t philox_seed,
                               uint64_t philox_counter, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!valid || !actions_out) return ML2048_E_NULL;
    if (misaligned(valid, 4)) return ML2048_E_ALIGN;
    const unsigned grid = (unsigned)((num_games + kStepThreads - 1) / kStepThreads);
    clear_stale_error();
    sample_random_valid_kernel<<<grid, kStepThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const uint32_t *>(valid), actions_out, num_games, slot_base, philox_seed, philox_counter);
    return launch_status();
}

int ml2048_sample_masked_categorical(const float *logits, const void *valid, uint8_t *actions_u8, int64_t *actions_i64, float *log_prob,
                                     int64_t num_games, int64_t slot_base, uint64_t philox_seed, uint64_t philox_counter, void *stream)
{
    if (num_games <= 0) return ML2048_E_SIZE;
    if (!logits || !valid || (!actions_u8 && !actions_i64)) return ML2048_E_NULL;
    if (misaligned(logits, 16) || misaligned(valid, 4) || misaligned(actions_i64, 8) || misaligned(log_prob, 4)) return ML2048_E_ALIGN;
    const unsigned grid = (unsigned)((num_games + kStepThreads - 1) / kStepThreads);
    clear_stale_error();
    sample_categorical_kernel<<<grid, kStepThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const float4 *>(logits), reinterpret_cast<const uint32_t *>(valid), actions_u8,
        reinterpret_cast<long long *>(actions_i64), log_prob, num_games, slot_base, philox_seed, philox_counter);
    return launch_status();
}

int ml2048_gae(const float *v0, const float *v1, const float *reward, const uint8_t *terminated, float *adv, int64_t use_count,
               int64_t step_count, int64_t game_count, float gamma, float coef, void *stream)
{
    if (use_count <= 0 || step_count <= 0 || game_count <= 0) return ML2048_E_SIZE;
    if (!v0 || !v1 || !reward || !terminated || !adv) return ML2048_E_NULL;
    if (misaligned(v0, 4) || misaligned(v1, 4) || misaligned(reward, 4) || misaligned(adv, 4)) return ML2048_E_ALIGN;
    const int64_t total = use_count * game_count;
    const unsigned grid = (unsigned)((total + kStepThreads - 1) / kStepThreads);
    clear_stale_error();
    gae_kernel<<<grid, kStepThreads, 0, static_cast<cudaStream_t>(stream)>>>(v0, v1, reward, terminated, adv, step_count, game_count,
                                                                            total, gamma, coef);
    return launch_status();
}

// Thin wrappers for host callers that drive the library without a CUDA binding of their own (the NumPy surface of VecGame at
// the training shape, where a framework-level copy + synchronise costs more host time than the kernels take).
int ml2048_copy_async(void *dst, const void *src, int64_t bytes, void *stream)
{
    if (!dst || !src) return ML2048_E_NULL;
    if (bytes <= 0) return ML2048_E_SIZE;
    return (int)cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDefault, static_cast<cudaStream_t>(stream));
}

int ml2048_stream_wait(void *stream) { return (int)cudaStreamSynchronize(static_cast<cudaStream_t>(stream)); }

uint32_t ml2048_two_mask(const float *host_randfloat16, double two_prob)
{
    // game_numba.py:207: `randfloat[idx] < two_prob` with idx the CELL index, f32 promoted to f64
    uint32_t m = 0;
    if (!host_randfloat16) return 0;
    for (int c = 0; c < 16; ++c)
        if ((double)host_randfloat16[c] < two_prob) m |= 1u << c;
    return m;
}

int ml2048_pack_randperm_keys(const uint8_t *host_randperm, uint8_t *host_keys, int64_t rows)
{
    // inverse form of each permutation row: keys[row][cell] = 16 * rank(cell) + cell, where rank(cell) is the
    // position of `cell` in the row, i.e. the order in which _spawn2 (game_numba.py:198-204) visits it
    if (!host_randperm || !host_keys) return ML2048_E_NULL;
    if (rows <= 0) return ML2048_E_SIZE;
    for (int64_t r = 0; r < rows; ++r) {
        const uint8_t *p = host_randperm + 16 * r;
        uint8_t *k = host_keys + 16 * r;
        unsigned seen = 0;
        for (int i = 0; i < 16; ++i) {
            if (p[i] > 15) return ML2048_E_ENUM;
            seen |= 1u << p[i];
            k[p[i]] = (uint8_t)(16 * i + p[i]);
        }
        if (seen != 0xffffu) return ML2048_E_ENUM;  // not a permutation of 0..15
    }
    return 0;
}

// host Philox (plain C++ copies of the rounds in board_ops.cuh, which are device functions in this translation unit)
static void host_philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1)
{
    for (int i = 0; i < 10; ++i) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        c[0] = n0, c[1] = (uint32_t)p1, c[2] = n2, c[3] = (uint32_t)p0;
        k0 += 0x9E3779B9u, k1 += 0xBB67AE85u;
    }
}

void ml2048_philox4x32_10(const uint32_t counter[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c[4] = {counter[0], counter[1], counter[2], counter[3]};
    host_philox4x32_10(c, key[0], key[1]);
    for (int i = 0; i < 4; ++i) out[i] = c[i];
}

void ml2048_philox2x32_10(const uint32_t counter[2], uint32_t key, uint32_t out[2])
{
    uint32_t c0 = counter[0], c1 = counter[1];
    for (int i = 0; i < 10; ++i) {
        const uint64_t p = (uint64_t)0xD256D193u * c0;
        c0 = (uint32_t)(p >> 32) ^ key ^ c1;
        c1 = (uint32_t)p;
        key += 0x9E3779B9u;
    }
    out[0] = c0, out[1] = c1;
}

void ml2048_philox_epoch_draws(uint64_t philox_seed, uint64_t prepare_counter, double two_prob, uint32_t *coin_u32, uint32_t *mask16)
{
    // counter words: (prepare counter low, high, stream tag, block index); key = seed
    const uint32_t k0 = (uint32_t)philox_seed, k1 = (uint32_t)(philox_seed >> 32);
    uint32_t c[4] = {(uint32_t)prepare_counter, (uint32_t)(prepare_counter >> 32), 0x434F494Eu /* "COIN" */, 0u};
    host_philox4x32_10(c, k0, k1);
    if (coin_u32) *coin_u32 = c[0];
    if (mask16) {
        const uint32_t thr = ml2048_two_threshold(two_prob);
        uint32_t m = 0;
        for (uint32_t b = 0; b < 4; ++b) {
            uint32_t w[4] = {(uint32_t)prepare_counter, (uint32_t)(prepare_counter >> 32), 0x4D41534Bu /* "MASK" */, b};
            host_philox4x32_10(w, k0, k1);
            for (uint32_t j = 0; j < 4; ++j)
                if (two_prob >= 1.0 || w[j] < thr) m |= 1u << (4 * b + j);
        }
        *mask16 = two_prob > 0.0 ? m : 0u;
    }
}

uint32_t ml2048_two_threshold(double two_prob)
{
    if (!(two_prob > 0.0)) return 0u;
    if (two_prob >= 1.0) return 0xffffffffu;
    return (uint32_t)(two_prob * 4294967296.0);
}

}  // extern "C"
