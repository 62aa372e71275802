// board_ops.cuh -- register-resident 2048 board arithmetic for sm_100a.
//
// A board is four 32-bit words (one per row), one byte per cell holding the tile exponent
// (0 = empty), cell = row*4+col with column 0 in the least significant byte -- i.e. exactly the 16
// bytes of the reference's `board` field read as a little-endian uint4 (game_numba.py:13-20, :542).
//
// Everything here is branch-free byte-SWAR on those words.  The move works "lane-parallel": the four
// lines that a move pushes are held as four words A,B,C,D where byte lane i belongs to line i and A is
// the cell next to the wall, so ONE sequence of 32-bit logic ops pushes all four lines at once.
// PRMT does the data movement (4x4 byte transpose) and, in its sign-replicating form, turns per-byte
// flags into full-byte masks; per-byte zero tests are carry-free adds (cells are <= 17 and xors of
// cells <= 31, so `byte + 0x7f` never carries into the next byte).  No local memory, no lookup tables.
//
// The header also compiles as plain C++ (tests/host_shim) so the arithmetic can be checked exhaustively
// against the CPU oracle without a GPU; the #else branch below emulates the four intrinsics it uses.
#pragma once
#include <stdint.h>
#if !defined(__CUDACC__)
#include <math.h>  // expf / logf / fmaxf of the sampler; included here because <cmath> breaks when first opened inside the namespace
#endif

#if defined(__CUDACC__)
#define ML2048_FN __device__ __forceinline__
#else
#define ML2048_FN static inline
#endif

namespace ml2048 {

#if defined(__CUDACC__)
ML2048_FN uint32_t prmt(uint32_t a, uint32_t b, uint32_t s) { return __byte_perm(a, b, s); }

// PRMT in its generic PTX form: a selector nibble with bit 3 set replicates the SIGN of the selected byte
// over the whole result byte (__byte_perm masks that bit away, so this needs inline PTX).
ML2048_FN uint32_t prmt_sign(uint32_t a, uint32_t b, uint32_t s)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(s));
    return d;
}
ML2048_FN uint32_t popc32(uint32_t x) { return (uint32_t)__popc(x); }
ML2048_FN uint32_t ffs32(uint32_t x) { return (uint32_t)__ffs((int)x); }
ML2048_FN uint32_t umulhi32(uint32_t a, uint32_t b) { return __umulhi(a, b); }
// min over three pairs of unsigned 16-bit lanes (DPX, one instruction on sm_90+)
ML2048_FN uint32_t min3_u16x2(uint32_t a, uint32_t b, uint32_t c) { return __vimin3_u16x2(a, b, c); }
ML2048_FN uint32_t max3_u16x2(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_u16x2(a, b, c); }
// 1 << (s mod 32): the funnel shift in wrap mode reads only the low five bits of s, so a byte of a packed word
// can be used as a shift count without masking it first
ML2048_FN uint32_t one_shl_wrap(uint32_t s) { return __funnelshift_l(0u, 1u, s); }
#else
ML2048_FN uint32_t prmt_sign(uint32_t a, uint32_t b, uint32_t s)
{
    const uint64_t pool = ((uint64_t)b << 32) | a;
    uint32_t d = 0;
    for (int i = 0; i < 4; ++i) {
        const uint32_t sel = (s >> (4 * i)) & 0xfu;
        uint32_t byte = (uint32_t)(pool >> (8 * (sel & 7u))) & 0xffu;
        if (sel & 8u) byte = (byte & 0x80u) ? 0xffu : 0x00u;
        d |= byte << (8 * i);
    }
    return d;
}
ML2048_FN uint32_t prmt(uint32_t a, uint32_t b, uint32_t s) { return prmt_sign(a, b, s & 0x7777u); }
ML2048_FN uint32_t popc32(uint32_t x) { return (uint32_t)__builtin_popcount(x); }
ML2048_FN uint32_t ffs32(uint32_t x) { return (uint32_t)__builtin_ffs((int)x); }
ML2048_FN uint32_t umulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
ML2048_FN uint32_t one_shl_wrap(uint32_t s) { return 1u << (s & 31u); }
ML2048_FN uint32_t max3_u16x2(uint32_t a, uint32_t b, uint32_t c)
{
    auto mx = [](uint32_t x, uint32_t y) { return x > y ? x : y; };
    const uint32_t lo = mx(mx(a & 0xffffu, b & 0xffffu), c & 0xffffu);
    const uint32_t hi = mx(mx(a >> 16, b >> 16), c >> 16);
    return lo | (hi << 16);
}
ML2048_FN uint32_t min3_u16x2(uint32_t a, uint32_t b, uint32_t c)
{
    auto mn = [](uint32_t x, uint32_t y) { return x < y ? x : y; };
    const uint32_t lo = mn(mn(a & 0xffffu, b & 0xffffu), c & 0xffffu);
    const uint32_t hi = mn(mn(a >> 16, b >> 16), c >> 16);
    return lo | (hi << 16);
}
#endif

// The step kernel saturates the integer ALU pipe (LOP3/PRMT/SHF/IADD: 84 % busy in ncu) while the FMA pipe
// idles (15 %).  An add written as `a * one + b` with a multiplier the compiler cannot see through is issued
// as IMAD on the FMA pipe; `one` lives in constant memory (an IMAD operand can come straight from there).
// The same goes for `a * 2^k + b` (a left shift, or a scaled add) and for `x & 0x01010101` of a full-byte mask x (bytes 0x00 /
// 0xff): x = 255 * e with e the 0/1 bytes, and 255 is odd, so e = x * 255^-1 = x * 0xfefefeff (mod 2^32) -- one IMAD computes
// `a + (x & 0x01010101)`.
#if defined(__CUDACC__)
__constant__ uint32_t c_opaque_one = 1u;
__constant__ uint32_t c_opaque_two = 2u;
__constant__ uint32_t c_opaque_256 = 256u;
__constant__ uint32_t c_opaque_2p23 = 0x00800000u;
__constant__ uint32_t c_opaque_inv255 = 0xfefefeffu;
// The multiply-add is written as PTX so that the front end cannot rewrite around it: it turned `~(a * one + b)` into
// `(-a) * one + ~b`, a negation (one more instruction) where the NOT would have been free inside the LOP3 that consumes it.
ML2048_FN uint32_t mad_opaque(uint32_t a, uint32_t m, uint32_t b)
{
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(m), "r"(b));
    return d;
}
ML2048_FN uint32_t add_on_fma_pipe(uint32_t a, uint32_t b) { return mad_opaque(a, c_opaque_one, b); }
ML2048_FN uint32_t twice_plus_on_fma_pipe(uint32_t a, uint32_t b) { return mad_opaque(a, c_opaque_two, b); }
ML2048_FN uint32_t shl8_on_fma_pipe(uint32_t a) { return mad_opaque(a, c_opaque_256, 0u); }
ML2048_FN uint32_t shl23_on_fma_pipe(uint32_t a) { return mad_opaque(a, c_opaque_2p23, 0u); }
ML2048_FN uint32_t add_ones_of_mask_on_fma_pipe(uint32_t a, uint32_t mask) { return mad_opaque(mask, c_opaque_inv255, a); }
ML2048_FN float bits_as_float(uint32_t x) { return __uint_as_float(x); }
#else
ML2048_FN uint32_t add_on_fma_pipe(uint32_t a, uint32_t b) { return a + b; }
ML2048_FN uint32_t twice_plus_on_fma_pipe(uint32_t a, uint32_t b) { return a * 2u + b; }
ML2048_FN uint32_t shl8_on_fma_pipe(uint32_t a) { return a << 8; }
ML2048_FN uint32_t shl23_on_fma_pipe(uint32_t a) { return a << 23; }
ML2048_FN uint32_t add_ones_of_mask_on_fma_pipe(uint32_t a, uint32_t mask) { return mask * 0xfefefeffu + a; }
ML2048_FN float bits_as_float(uint32_t x)
{
    float f;
    __builtin_memcpy(&f, &x, 4);
    return f;
}
#endif

constexpr uint32_t kHi = 0x80808080u;
constexpr uint32_t kLo7 = 0x7f7f7f7fu;
constexpr uint32_t kOnes = 0x01010101u;

// bit 7 of every byte set iff the cell is non-empty (the other bits are leftovers of the add)
ML2048_FN uint32_t occupied_signs(uint32_t row) { return add_on_fma_pipe(row, kLo7); }

// 0x80 in every byte whose cell is non-empty
ML2048_FN uint32_t occupied_flags(uint32_t row) { return occupied_signs(row) & kHi; }

// 0xff in every byte of x that is non-zero (bytes of x must be <= 0x80)
ML2048_FN uint32_t nonzero_mask(uint32_t x) { return prmt_sign(add_on_fma_pipe(x, kLo7), 0u, 0xba98); }

// What one move fused: `first`/`second` hold, one byte per line, the exponent of the consumed tiles PLUS 127 (0 = no fusion;
// a line fuses at most twice).  The bias makes a byte the exponent field of the float 2^k (bit 7 doubles as the "fused"
// flag, the low five bits are k - 1), which is how fusion_gain sums the rewards on the FMA pipe.  From them: the
// reference's reward_fn_normal (game_numba.py:408-438), reward_fn_rank (:469-484), the merged.sum() of reward_fn_maxcell
// (:502) and the `merged` array itself.
struct Fusions {
    uint32_t first;
    uint32_t second;
};

// number of fusions of the move (<= 8)
ML2048_FN uint32_t fusion_count(const Fusions &f) { return popc32(f.first & kHi) + popc32(f.second & kHi); }

// Four lines pushed toward A at once.  Same result per line as the reference's _push_row
// (game_numba.py:48-90): stable compaction of the tiles, then equal neighbours fuse once, in order
// from the wall, a fused tile never fusing again.
ML2048_FN void push4(uint32_t &A, uint32_t &B, uint32_t &C, uint32_t &D, Fusions &f)
{
    // stable compaction: close the gap at position C, then B, then A
    uint32_t m;
    m = nonzero_mask(C);
    C = C | (D & ~m);
    D = D & m;
    m = nonzero_mask(B);
    B = B | (C & ~m);
    C = (C & m) | (D & ~m);
    D = D & m;
    m = nonzero_mask(A);
    A = A | (B & ~m);
    B = (B & m) | (C & ~m);
    C = (C & m) | (D & ~m);
    D = D & m;
    // which neighbours fuse (full-byte masks): a/b first, then b/c unless b was used, then c/d unless c was used
    const uint32_t sA = add_on_fma_pipe(A, kLo7), sB = add_on_fma_pipe(B, kLo7), sC = add_on_fma_pipe(C, kLo7);  // cell + 127
    const uint32_t eab = ~nonzero_mask(A ^ B) & prmt_sign(sA, 0u, 0xba98);
    const uint32_t ebc = ~nonzero_mask(B ^ C) & prmt_sign(sB, 0u, 0xba98) & ~eab;
    const uint32_t ecd = ~nonzero_mask(C ^ D) & prmt_sign(sC, 0u, 0xba98) & ~ebc;
    f.first = (sA & eab) | (sB & ebc) | (sC & ecd & ~eab);  // per line these three exclude each other
    f.second = sC & ecd & eab;
    const uint32_t both = eab & ecd;    // [a+1, c+1, 0, 0]
    const uint32_t shift = eab | ebc;   // position C receives D
    const uint32_t nA = add_ones_of_mask_on_fma_pipe(A, eab);
    const uint32_t nB = add_ones_of_mask_on_fma_pipe((C & eab) | (B & ~eab), ebc | both);
    const uint32_t nC = (D & shift & ~both) | (add_ones_of_mask_on_fma_pipe(C, ecd) & ~shift);
    const uint32_t nD = D & ~(shift | ecd);
    A = nA, B = nB, C = nC, D = nD;
}

// sum over the (up to 8) fusions of 2^(k+1): the reference's reward_fn_normal, as the float the reward and the score are
// (exact: every term is a power of two <= 2^18 and the sum stays below 2^22).  A candidate byte v = k + 127 shifted into the
// exponent field IS the float 2^k, and v = 0 is 0.0f: one byte extraction (ALU pipe) per candidate, the shift as a multiply
// and the sum on the FMA pipe -- the integer version (eight variable shifts and their adds) cost 21 ALU-pipe instructions.
ML2048_FN float fusion_gain(const Fusions &f)
{
    float s = bits_as_float(shl23_on_fma_pipe(f.first & 0xffu)) + bits_as_float(shl23_on_fma_pipe(f.second & 0xffu));
    s += bits_as_float(shl23_on_fma_pipe(prmt(f.first, 0u, 0x4441))) + bits_as_float(shl23_on_fma_pipe(prmt(f.second, 0u, 0x4441)));
    s += bits_as_float(shl23_on_fma_pipe(prmt(f.first, 0u, 0x4442))) + bits_as_float(shl23_on_fma_pipe(prmt(f.second, 0u, 0x4442)));
    s += bits_as_float(shl23_on_fma_pipe(prmt(f.first, 0u, 0x4443))) + bits_as_float(shl23_on_fma_pipe(prmt(f.second, 0u, 0x4443)));
    return s + s;
}

// sum over the fusions of (k+1): reward_fn_rank.  (v & 31) = k - 1 for a fused candidate, 0 otherwise.
ML2048_FN uint32_t fusion_rank(const Fusions &f)
{
    return ((((f.first & 0x1f1f1f1fu) + (f.second & 0x1f1f1f1fu)) * kOnes) >> 24) + 2u * fusion_count(f);
}

// the reference's `merged` u8[16] as four words: merged[k] = number of fusions that consumed exponent k.
// Exponents >= 16 have no slot (game_numba.py:543; the reference would index out of bounds) and are dropped.
ML2048_FN void fusion_log(const Fusions &f, uint32_t &m0, uint32_t &m1, uint32_t &m2, uint32_t &m3)
{
    unsigned long long nib = 0ull;  // sixteen 4-bit counters
    const uint32_t w[2] = {f.first, f.second};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t v = (w[i] >> (8 * j)) & 0xffu;
            const uint32_t k = (v & 0x1fu) + 1u;
            if (v != 0u && k < 16u) nib += 1ull << (4u * k);
        }
    }
    const uint32_t lo = (uint32_t)nib, hi = (uint32_t)(nib >> 32);
    m0 = lo & 0xffffu, m1 = lo >> 16, m2 = hi & 0xffffu, m3 = hi >> 16;
    m0 = (m0 | (m0 << 8)) & 0x00ff00ffu; m0 = (m0 | (m0 << 4)) & 0x0f0f0f0fu;
    m1 = (m1 | (m1 << 8)) & 0x00ff00ffu; m1 = (m1 | (m1 << 4)) & 0x0f0f0f0fu;
    m2 = (m2 | (m2 << 8)) & 0x00ff00ffu; m2 = (m2 | (m2 << 4)) & 0x0f0f0f0fu;
    m3 = (m3 | (m3 << 8)) & 0x00ff00ffu; m3 = (m3 | (m3 << 4)) & 0x0f0f0f0fu;
}

// The move itself: direction dispatch of _step_kernel (game_numba.py:93-134) without a branch AND without selects.
// The lines a move pushes reach push4 through a two-stage byte-permute network (PRMT takes its selector from a
// register), and the pushed words go back to rows through a second one; what differs between the four directions is
// only the six selectors: for UP/DOWN the network passes the rows through (in reverse order for DOWN), for LEFT/RIGHT it
// is the 4x4 byte transpose (with the columns taken in reverse order for RIGHT).  One 32-byte row of this table per
// action: {in1a, in1b, in2a, in2b, out2a, out2b, 0, 0}; the step kernel keeps the table in global memory (L1) and fetches a
// game's row with two vector loads instead of deciding per word with compare + select (16 SEL per move before).
//   stage 1: t0 = P(r0,r2,in1a) t1 = P(r1,r3,in1a) t2 = P(r0,r2,in1b) t3 = P(r1,r3,in1b)
//   stage 2: A = P(t0,t1,in2a) B = P(t0,t1,in2b) C = P(t2,t3,in2a) D = P(t2,t3,in2b)
//   back   : u0 = P(A,C,in2a) u1 = P(B,D,in2a) u2 = P(A,C,in2b) u3 = P(B,D,in2b)
//            r0 = P(u0,u1,out2a) r1 = P(u0,u1,out2b) r2 = P(u2,u3,out2a) r3 = P(u2,u3,out2b)
constexpr int kMoveSelRow = 8;  // words per action
#define ML2048_MOVE_SEL_TABLE                                                     \
    {                                                                             \
        0x5140u, 0x7362u, 0x5140u, 0x7362u, 0x5140u, 0x7362u, 0u, 0u, /* left  */ \
        0x6273u, 0x4051u, 0x5140u, 0x7362u, 0x0415u, 0x2637u, 0u, 0u, /* right */ \
        0x3210u, 0x7654u, 0x3210u, 0x7654u, 0x3210u, 0x7654u, 0u, 0u, /* up    */ \
        0x7654u, 0x3210u, 0x7654u, 0x3210u, 0x7654u, 0x3210u, 0u, 0u  /* down  */ \
    }

// The same rows indexed by (valid-direction mask, k): row 4*bits + k holds the selectors of the k-th (0-based) valid direction
// of the 4-bit mask `bits` and, in word 6, that direction itself.  The in-kernel random policy picks k = floor(u * popc(bits))
// and fetches the row directly: no search for the k-th set bit (16 ALU instructions before).  Rows 60..63 (bits = 0b1111)
// are the four directions in order, i.e. the table a caller-given action indexes with 60 + action; k beyond the number of
// valid directions (only reachable with bits = 0, a finished game idling) maps to direction 0.
struct PolicySelTable {
    uint32_t w[64 * kMoveSelRow];
};

constexpr PolicySelTable make_policy_sel_table()
{
    constexpr uint32_t base[4 * kMoveSelRow] = ML2048_MOVE_SEL_TABLE;
    PolicySelTable t{};
    for (uint32_t bits = 0; bits < 16; ++bits) {
        for (uint32_t k = 0; k < 4; ++k) {
            uint32_t action = 0, seen = 0;
            bool found = false;
            for (uint32_t d = 0; d < 4 && !found; ++d) {
                if ((bits >> d) & 1u) {
                    if (seen == k) {
                        action = d;
                        found = true;
                    }
                    ++seen;
                }
            }
            for (int j = 0; j < kMoveSelRow; ++j) t.w[(4 * bits + k) * kMoveSelRow + j] = base[action * kMoveSelRow + j];
            t.w[(4 * bits + k) * kMoveSelRow + 6] = action;
        }
    }
    return t;
}

// The move with its row of the table already fetched: words 0..3 in `sa`, 4..6 in `sb`.
// Returns word 6 of the row (the direction, in the (mask, k)-indexed table).
struct SelRow {
    uint32_t in1a, in1b, in2a, in2b, out2a, out2b, action;
};

ML2048_FN uint32_t move_board_row(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, const SelRow &s, Fusions &f)
{
    // prmt_sign = the raw PRMT (no selector nibble of the table has its sign-replication bit set); __byte_perm would
    // first mask a selector it cannot see to 0x7777
    const uint32_t t0 = prmt_sign(r0, r2, s.in1a), t1 = prmt_sign(r1, r3, s.in1a), t2 = prmt_sign(r0, r2, s.in1b), t3 = prmt_sign(r1, r3, s.in1b);
    uint32_t A = prmt_sign(t0, t1, s.in2a), B = prmt_sign(t0, t1, s.in2b), C = prmt_sign(t2, t3, s.in2a), D = prmt_sign(t2, t3, s.in2b);
    push4(A, B, C, D, f);
    const uint32_t u0 = prmt_sign(A, C, s.in2a), u1 = prmt_sign(B, D, s.in2a), u2 = prmt_sign(A, C, s.in2b), u3 = prmt_sign(B, D, s.in2b);
    r0 = prmt_sign(u0, u1, s.out2a);
    r1 = prmt_sign(u0, u1, s.out2b);
    r2 = prmt_sign(u2, u3, s.out2a);
    r3 = prmt_sign(u2, u3, s.out2b);
    return s.action;
}

// `sel` = the action's row of the table in GLOBAL memory (16-byte aligned)
ML2048_FN uint32_t move_board_sel(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, const uint32_t *sel, Fusions &f)
{
#if defined(__CUDACC__)
    const uint4 sa = __ldg(reinterpret_cast<const uint4 *>(sel));
    const uint4 sb = __ldg(reinterpret_cast<const uint4 *>(sel + 4));
    const SelRow row{sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z};
#else
    const SelRow row{sel[0], sel[1], sel[2], sel[3], sel[4], sel[5], sel[6]};
#endif
    return move_board_row(r0, r1, r2, r3, row, f);
}

#if !defined(__CUDACC__)
// host build (tests/host_shim): the table is a plain static array
ML2048_FN void move_board(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, uint32_t action, Fusions &f)
{
    static const uint32_t table[4 * kMoveSelRow] = ML2048_MOVE_SEL_TABLE;
    move_board_sel(r0, r1, r2, r3, table + (action & 3u) * kMoveSelRow, f);
}
#endif

// Valid-action mask, one byte per direction (left,right,up,down), as the little-endian word the
// reference stores in `valid_actions` (game_numba.py:259-289).  A direction is valid iff some tile
// can slide into an empty cell or fuse with its neighbour on that axis -- the predicate
// _line_movable (:215-256) enumerates pairwise, proven equal to "the move changes the board" for
// all 18^4 lines (tests/test_oracle_golden.py::test_line_table_exhaustive).
//   slide toward a wall  <=>  some tile has an EMPTY neighbour on the wall side
//   fuse on an axis      <=>  some tile equals its neighbour on that axis
ML2048_FN uint32_t valid_mask(uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3)
{
    const uint32_t s0 = occupied_signs(r0), s1 = occupied_signs(r1), s2 = occupied_signs(r2), s3 = occupied_signs(r3);
    // Slides on ONE packed word P: byte j = column j, bit 7-i of it = "row i holds a tile".  Each row's flag is born at its own
    // bit position by a scaled add (cells are <= 17): c + 0x7f sets bit 7, 2c + 0x3e bit 6, c + 0x1f bit 5 exactly when c >= 1;
    // for bit 4, c + 0x0f covers 1..16 and the cell's own bit 4 covers 16 and 17.  The adds are FMA-pipe work; three LOP3 merge them.
    const uint32_t x1 = twice_plus_on_fma_pipe(r1, 0x3e3e3e3eu), x2 = add_on_fma_pipe(r2, 0x1f1f1f1fu), x3 = add_on_fma_pipe(r3, 0x0f0f0f0fu);
    const uint32_t t3 = (x3 | r3) & 0x10101010u;
    const uint32_t P = (s0 & kHi) | (x1 & 0x40404040u) | (x2 & 0x20202020u) | t3;
    const uint32_t Pr = P >> 8;                    // byte j = column j + 1
    const uint32_t Pl = shl8_on_fma_pipe(P);       // byte j = column j - 1
    const uint32_t Pd = twice_plus_on_fma_pipe(P, 0u);  // bit 7-i = row i + 1 (bit 0 of a byte catches the neighbour's bit 7: masked below)
    // fusions: xor of neighbours is zero where the first one is a tile (byte 3 of a row xor is the cell itself)
    const uint32_t hfuse = ((~add_on_fma_pipe(r0 ^ (r0 >> 8), kLo7) & s0) | (~add_on_fma_pipe(r1 ^ (r1 >> 8), kLo7) & s1) |
                            (~add_on_fma_pipe(r2 ^ (r2 >> 8), kLo7) & s2) | (~add_on_fma_pipe(r3 ^ (r3 >> 8), kLo7) & s3)) & kHi;
    const uint32_t vfuse = (~add_on_fma_pipe(r0 ^ r1, kLo7) & s0) | (~add_on_fma_pipe(r1 ^ r2, kLo7) & s1) |
                           (~add_on_fma_pipe(r2 ^ r3, kLo7) & s2);
    const bool vf = (vfuse & kHi) != 0u;
    // a tile at column j+1 next to an empty column j can slide left, and so on
    const uint32_t l = (((Pr & ~P) | hfuse) != 0u) ? 1u : 0u;
    const uint32_t r = (((Pl & ~P) | hfuse) != 0u) ? 1u : 0u;
    const uint32_t u = (((Pd & ~P & 0xe0e0e0e0u) != 0u) || vf) ? 1u : 0u;
    const uint32_t d = (((P & ~Pd & 0xe0e0e0e0u) != 0u) || vf) ? 1u : 0u;
    return (l + r * 0x100u) + (u * 0x10000u + d * 0x1000000u);  // disjoint bytes: adds (IMAD) instead of shifts + ORs
}

// Write `value` (a tile exponent, or any small multiplier) into cell `cell` (0..15) of the (empty there) board.  The sixteen
// boards with a single 1 live in a 256-byte table (L1-resident): one vector load and four multiply-adds on the FMA pipe
// instead of a 64-bit shift and four selects (14 ALU-pipe instructions with the 2-or-4 decision; 4 now).
struct CellTable {
    uint32_t w[16 * 4];
};

constexpr CellTable make_cell_table()
{
    CellTable t{};
    for (uint32_t c = 0; c < 16; ++c) t.w[4 * c + (c >> 2)] = 1u << (8u * (c & 3u));
    return t;
}

#if defined(__CUDACC__)
__device__ const CellTable d_cell_one = make_cell_table();
#endif

#if defined(__CUDACC__)
// ... with the cell's table entry already fetched
ML2048_FN void put_cell_entry(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, uint4 t, uint32_t value)
{
    r0 = t.x * value + r0;
    r1 = t.y * value + r1;
    r2 = t.z * value + r2;
    r3 = t.w * value + r3;
}
#endif

ML2048_FN void put_cell(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, uint32_t cell, uint32_t value)
{
#if defined(__CUDACC__)
    put_cell_entry(r0, r1, r2, r3, __ldg(reinterpret_cast<const uint4 *>(d_cell_one.w) + cell), value);
#else
    constexpr CellTable tab = make_cell_table();
    r0 += tab.w[4 * cell] * value;
    r1 += tab.w[4 * cell + 1] * value;
    r2 += tab.w[4 * cell + 2] * value;
    r3 += tab.w[4 * cell + 3] * value;
#endif
}

// The same without the table: one 64-bit shift places the value inside its half of the board, one predicate picks the half.
// For the latency-bound small-batch kernels, where a dependent load from a cold table costs more than ten ALU instructions.
ML2048_FN void put_cell_shift(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, uint32_t cell, uint32_t value)
{
    const unsigned long long v = (unsigned long long)value << ((cell & 7u) * 8u);
    const uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
    const bool top = (cell & 8u) != 0u;
    r0 += top ? 0u : lo;
    r1 += top ? 0u : hi;
    r2 += top ? lo : 0u;
    r3 += top ? hi : 0u;
}

// Replay-mode spawn position.  The reference walks row `p` of randperm and takes the first entry whose
// cell is empty (_spawn2, game_numba.py:198-204).  Equivalently: among the empty cells take the one with
// the smallest RANK in that row.  `keys` is the row in inverse form, keys[c] = 16*rank(c) + c (see
// ml2048_pack_randperm_keys); one min-reduction over the sixteen keys (as 16-bit lanes, DPX three-input
// min), with occupied cells pushed out of range, yields the winner.  Returns the cell, or 16 if the board is full.
// n0..n3: bit 7 of every byte set iff the cell is occupied; the other bits are ignored (so `row + 0x7f7f7f7f` will do).
ML2048_FN uint32_t first_empty_key(uint32_t k0, uint32_t k1, uint32_t k2, uint32_t k3, uint32_t n0, uint32_t n1, uint32_t n2,
                                   uint32_t n3)
{
    // widen every key byte to a 16-bit lane whose HIGH byte is 0xff when the cell is occupied (one PRMT takes the key
    // byte and replicates the sign of the occupancy byte next to it), so any occupied lane (>= 0xff00) loses against
    // any empty one (<= 0x00ff)
    const uint32_t a0 = prmt_sign(k0, n0, 0xd1c0), a1 = prmt_sign(k0, n0, 0xf3e2);
    const uint32_t b0 = prmt_sign(k1, n1, 0xd1c0), b1 = prmt_sign(k1, n1, 0xf3e2);
    const uint32_t c0 = prmt_sign(k2, n2, 0xd1c0), c1 = prmt_sign(k2, n2, 0xf3e2);
    const uint32_t d0 = prmt_sign(k3, n3, 0xd1c0), d1 = prmt_sign(k3, n3, 0xf3e2);
    const uint32_t m = min3_u16x2(min3_u16x2(a0, a1, b0), min3_u16x2(b1, c0, c1), min3_u16x2(d0, d1, d1));
    // both halves of the result = the smaller half: its low byte is the winning key (low nibble = the cell), its high
    // byte is 0xff iff the board is full
    return min3_u16x2(m, prmt(m, 0u, 0x1032), m);
}

// The cell (0..15), or 16 if the board is full.
ML2048_FN uint32_t first_empty_by_rank(uint32_t k0, uint32_t k1, uint32_t k2, uint32_t k3, uint32_t n0, uint32_t n1,
                                       uint32_t n2, uint32_t n3)
{
    const uint32_t m = first_empty_key(k0, k1, k2, k3, n0, n1, n2, n3) & 0xffffu;
    return m >= 0xff00u ? 16u : (m & 15u);
}

// 16-bit mask of empty cells from the per-row 0x80 "empty" flags (multiply gathers bits 7,15,23,31 into a nibble)
ML2048_FN uint32_t empties16(uint32_t z0, uint32_t z1, uint32_t z2, uint32_t z3)
{
    const uint32_t m = 0x00204081u;
    return ((z0 * m) >> 28) | (((z1 * m) >> 24) & 0xf0u) | (((z2 * m) >> 20) & 0xf00u) | (((z3 * m) >> 16) & 0xf000u);
}

// index of the k-th (0-based) set bit of a 16-bit mask; k < popc(mask)
ML2048_FN uint32_t kth_set_bit16(uint32_t mask, uint32_t k)
{
    uint32_t pos = 0u, c;
    c = popc32(mask & 0xffu);
    if (k >= c) { k -= c; pos = 8u; mask >>= 8; }
    c = popc32(mask & 0xfu);
    if (k >= c) { k -= c; pos += 4u; mask >>= 4; }
    c = popc32(mask & 0x3u);
    if (k >= c) { k -= c; pos += 2u; mask >>= 2; }
    c = mask & 1u;
    if (k >= c) { pos += 1u; }
    return pos;
}

// The four 0/1 bytes of a valid-action word (left,right,up,down) as a 4-bit mask (multiply gathers bits 0,8,16,24)
ML2048_FN uint32_t mask_bits4(uint32_t valid_word) { return (valid_word * 0x10204080u) >> 28; }

// k-th (0-based) valid direction of a 4-bit mask, k < popc(bits): strip the k lowest set bits, take the next one
ML2048_FN uint32_t kth_valid_action(uint32_t bits, uint32_t k)
{
    uint32_t t = bits;
    t = (k > 0u) ? (t & (t - 1u)) : t;
    t = (k > 1u) ? (t & (t - 1u)) : t;
    t = (k > 2u) ? (t & (t - 1u)) : t;
    return ffs32(t) - 1u;
}

// max tile exponent of a board: the sixteen bytes as sixteen 16-bit lanes (even and odd bytes of every row: one mask / one
// byte permute each) and a three-input lane-wise max (DPX, VIMNMX3.U16x2) down to one word: 15 instructions (24 with byte-wise
// compare-and-select)
ML2048_FN uint32_t max_cell(uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3)
{
    const uint32_t e0 = r0 & 0x00ff00ffu, e1 = r1 & 0x00ff00ffu, e2 = r2 & 0x00ff00ffu, e3 = r3 & 0x00ff00ffu;
    const uint32_t o0 = prmt(r0, 0u, 0x4341), o1 = prmt(r1, 0u, 0x4341), o2 = prmt(r2, 0u, 0x4341), o3 = prmt(r3, 0u, 0x4341);
    const uint32_t m = max3_u16x2(max3_u16x2(e0, e1, e2), max3_u16x2(e3, o0, o1), max3_u16x2(o2, o3, o3));
    return max3_u16x2(m, m >> 16, m) & 0xffffu;
}

// Philox4x32-10 (Salmon et al., SC'11), counter-based: out = f(counter, key)
struct u32x4 {
    uint32_t x, y, z, w;
};

ML2048_FN u32x4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1)
{
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = umulhi32(M0, c0), lo0 = M0 * c0;
        const uint32_t hi1 = umulhi32(M1, c2), lo1 = M1 * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += W0;
        k1 += W1;
    }
    return u32x4{c0, c1, c2, c3};
}

// Every board a reset can produce: two tiles on an empty board (game_numba.py:648-655).  Entry
//   idx = (c0 << 6) | (c1 << 2) | (t0 << 1) | t1      c = cell of the first / second tile, t = 1 for a 2-tile, 0 for a 4-tile
// holds the board (four row words) and its valid-action word, so the auto-reset looks both up with two loads instead of
// building the board with 64-bit shifts and running the 75-instruction mask on it -- the fused auto-reset executes this
// once per WARP that holds a finished game (a quarter of all warps in steady state), so its length matters.
struct FreshTable {
    uint32_t board[1024 * 4];
    uint32_t mask[1024];
};

constexpr uint32_t scalar_valid_word(const uint8_t (&b)[16])
{
    bool l = false, r = false, u = false, d = false;
    for (int row = 0; row < 4; ++row) {
        for (int col = 0; col < 4; ++col) {
            const uint8_t x = b[4 * row + col];
            if (x == 0) continue;
            if (col > 0 && (b[4 * row + col - 1] == 0 || b[4 * row + col - 1] == x)) l = true;
            if (col < 3 && (b[4 * row + col + 1] == 0 || b[4 * row + col + 1] == x)) r = true;
            if (row > 0 && (b[4 * (row - 1) + col] == 0 || b[4 * (row - 1) + col] == x)) u = true;
            if (row < 3 && (b[4 * (row + 1) + col] == 0 || b[4 * (row + 1) + col] == x)) d = true;
        }
    }
    return (l ? 1u : 0u) | (r ? 0x100u : 0u) | (u ? 0x10000u : 0u) | (d ? 0x1000000u : 0u);
}

constexpr FreshTable make_fresh_table()
{
    FreshTable t{};
    for (uint32_t idx = 0; idx < 1024; ++idx) {
        const uint32_t c0 = idx >> 6, c1 = (idx >> 2) & 15u, t0 = (idx >> 1) & 1u, t1 = idx & 1u;
        uint8_t b[16] = {};
        b[c0] = (uint8_t)(2u - t0);
        b[c1] = (uint8_t)(b[c1] + (2u - t1));  // c0 == c1 cannot occur (distinct cells); an add like the kernel's put_cell
        for (int row = 0; row < 4; ++row)
            t.board[4 * idx + row] = (uint32_t)b[4 * row] | ((uint32_t)b[4 * row + 1] << 8) | ((uint32_t)b[4 * row + 2] << 16) |
                                     ((uint32_t)b[4 * row + 3] << 24);
        t.mask[idx] = scalar_valid_word(b);
    }
    return t;
}

// Philox2x32-10 (same family, Random123): two 32-bit words per block, half the multiplies and xors of Philox4x32-10.
// A game-step consumes two uniform words -- the spawn cell (Philox mode) and the policy's action -- so this is the block
// the kernels draw; the 4x32 variant serves the host-side epoch draws (ml2048_philox_epoch_draws).
struct u32x2 {
    uint32_t x, y;
};

ML2048_FN u32x2 philox2x32_10(uint32_t c0, uint32_t c1, uint32_t k)
{
    const uint32_t M = 0xD256D193u, W = 0x9E3779B9u;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi = umulhi32(M, c0), lo = M * c0;
        c0 = hi ^ k ^ c1;
        c1 = lo;
        k += W;
    }
    return u32x2{c0, c1};
}

// The same rounds with the ten round keys handed in (key + i * W): a kernel whose host code knows the seed passes them as
// kernel parameters, and the rounds then read them straight from the constant bank instead of deriving them once per warp.
struct PhiloxKeys {
    uint32_t k[10];
};

ML2048_FN u32x2 philox2x32_10_keys(uint32_t c0, uint32_t c1, const PhiloxKeys &keys)
{
    const uint32_t M = 0xD256D193u;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi = umulhi32(M, c0), lo = M * c0;
        c0 = hi ^ keys.k[i] ^ c1;
        c1 = lo;
    }
    return u32x2{c0, c1};
}

// One Philox2x32-10 block of stream `tag` (0 = the policy's words, kSpawnStream = the spawn cells of Philox mode, kResetStream
// = the auto-reset's two cells): counter = (index low word, counter low word ^ high words * odd constants), key = seed ^ tag.
// The key depends on nothing but the seed (a kernel parameter), so its ten round values are computed once per warp on the
// uniform datapath -- the step counter may come from a device-resident schedule entry, i.e. from a vector register, and a key
// built from it costs nine ALU adds per game-step.
constexpr uint32_t kResetStream = 0x80000000u;
constexpr uint32_t kSpawnStream = 0x40000000u;

ML2048_FN uint32_t stream_key(uint64_t seed, uint32_t tag) { return (uint32_t)seed ^ ((uint32_t)(seed >> 32) * 0x9E3779B9u) ^ tag; }

ML2048_FN uint32_t block_counter_word(uint64_t index, uint64_t counter)
{
    return (uint32_t)counter ^ ((uint32_t)(counter >> 32) * 0x85EBCA6Bu) ^ ((uint32_t)(index >> 32) * 0xC2B2AE35u);
}

ML2048_FN u32x2 slot_draws(uint64_t index, uint64_t counter, uint64_t seed, uint32_t tag)
{
    return philox2x32_10((uint32_t)index, block_counter_word(index, counter), stream_key(seed, tag));
}

// ... with the stream's round keys precomputed (philox_round_keys)
ML2048_FN u32x2 slot_draws_keys(uint64_t index, uint64_t counter, const PhiloxKeys &keys)
{
    return philox2x32_10_keys((uint32_t)index, block_counter_word(index, counter), keys);
}

ML2048_FN uint32_t slot_word_keys(uint64_t slot, uint64_t counter, const PhiloxKeys &keys)
{
    const u32x2 b = slot_draws_keys(slot >> 1, counter, keys);
    return (slot & 1ull) ? b.y : b.x;
}

inline PhiloxKeys philox_round_keys(uint64_t seed, uint32_t tag)  // host side
{
    PhiloxKeys keys;
    uint32_t k = (uint32_t)seed ^ ((uint32_t)(seed >> 32) * 0x9E3779B9u) ^ tag;  // stream_key
    for (int i = 0; i < 10; ++i, k += 0x9E3779B9u) keys.k[i] = k;
    return keys;
}

// The ONE uniform word a game-step takes from the policy stream (and, in Philox mode, from the spawn stream): a block holds
// two words, so it serves a PAIR of global slots -- block index = slot >> 1, the even slot takes .x, the odd one .y.  A thread
// that owns both slots of a pair (step_pair_kernel) computes the block once; draws stay a function of (seed, global slot,
// counter) alone, i.e. independent of batch size, sharding and kernel variant.
ML2048_FN uint32_t slot_word(uint64_t slot, uint64_t counter, uint64_t seed, uint32_t tag)
{
    const u32x2 b = slot_draws(slot >> 1, counter, seed, tag);
    return (slot & 1ull) ? b.y : b.x;
}

// Masked categorical sample (policy/actor_critic.py:56-76): invalid actions get finfo.min, the logits are
// normalised as torch's Categorical does (x - logsumexp(x), logsumexp = max + log(sum(exp(x - max)))), one
// uniform u in [0,1) picks the action by inverse CDF.  `mask_bits` bit k = action k valid.  Returns the action
// and its log-probability.  The host build (tests/host_shim) uses the C library's expf/logf, the device build CUDA's; both
// are checked against a float64 reference.
ML2048_FN uint32_t sample_masked_categorical(float l0, float l1, float l2, float l3, uint32_t mask_bits, uint32_t rnd,
                                             float &log_prob)
{
    const float kMin = -3.4028234663852886e38f;  // torch.finfo(float32).min
    l0 = (mask_bits & 1u) ? l0 : kMin;
    l1 = (mask_bits & 2u) ? l1 : kMin;
    l2 = (mask_bits & 4u) ? l2 : kMin;
    l3 = (mask_bits & 8u) ? l3 : kMin;
    const float mx = fmaxf(fmaxf(l0, l1), fmaxf(l2, l3));
    const float e0 = expf(l0 - mx), e1 = expf(l1 - mx), e2 = expf(l2 - mx), e3 = expf(l3 - mx);
    const float total = ((e0 + e1) + e2) + e3;
    const float lse = logf(total) + mx;
    const float t = (float)(rnd >> 8) * (1.0f / 16777216.0f) * total;
    const float c0 = e0, c1 = c0 + e1, c2 = c1 + e2;
    uint32_t action = (t < c0) ? 0u : (t < c1) ? 1u : (t < c2) ? 2u : 3u;
    // rounding may push t onto an impossible action (e == 0): fall back to the last possible one
    const float ea = action == 0u ? e0 : action == 1u ? e1 : action == 2u ? e2 : e3;
    if (ea == 0.0f) action = (e3 > 0.0f) ? 3u : (e2 > 0.0f) ? 2u : (e1 > 0.0f) ? 1u : 0u;
    const float la = action == 0u ? l0 : action == 1u ? l1 : action == 2u ? l2 : l3;
    log_prob = la - lse;
    return action;
}

// ---- n-tuple networks -----------------------------------------------------------------------
// K <= 16 tuples of 1..6 distinct cells; tuple t owns one float32 table of 16^len entries, all tables back to back in tuple
// order.  A board's value sums, for every tuple and each of the board's 8 symmetric images, the table entry indexed by the
// image's cells under the tuple: idx = sum_j min(cell_j, 15) << 4j.  Clamping makes every byte value an in-bounds index (the
// board is never trusted to stay below 16); tiles 2^16 (exponent 16) and above share the entries of 2^15.
constexpr int kNTupleMaxTuples = 16;
constexpr int kNTupleMaxLen = 6;

// Image g (0..7) of a board s holds in cell 4r+c the cell ntuple_sym_src(g, 4r+c) of s:
// (r,c) (r,3-c) (3-r,c) (3-r,3-c) (c,r) (c,3-r) (3-c,r) (3-c,3-r) -- bit 2 of g transposes, bit 1 flips rows, bit 0 columns.
#if defined(__CUDACC__)
__host__ __device__
#endif
constexpr uint32_t ntuple_sym_src(uint32_t g, uint32_t cell)
{
    const uint32_t r = cell >> 2, c = cell & 3u;
    const uint32_t rt = (g & 4u) ? c : r, ct = (g & 4u) ? r : c;
    return 4u * ((g & 2u) ? 3u - rt : rt) + ((g & 1u) ? 3u - ct : ct);
}

// The network as the kernels take it, by value (a kernel parameter: two networks in one process and CUDA-graph capture need
// no device symbol).  src4[t][g][j] = 4 * the ORIGINAL cell that image g puts under cell j of tuple t, i.e. the bit position of
// that cell's field in ntuple_nibbles.  offset[t] < 16 * 16^6 = 2^28: 32 bits hold every entry index.
struct NTupleSpec {
    uint32_t num_tuples;
    uint32_t len[kNTupleMaxTuples];
    uint32_t offset[kNTupleMaxTuples];
    uint8_t src4[kNTupleMaxTuples][8][8];  // rows padded to 8
};

// Host side: expand validated tuples (cells [K][6], len [K]) into the kernels' form.  Returns the total number of entries.
inline int64_t ntuple_expand(const uint8_t *cells, const uint8_t *len, int32_t num_tuples, NTupleSpec &s)
{
    s = NTupleSpec{};
    s.num_tuples = (uint32_t)num_tuples;
    int64_t total = 0;
    for (int t = 0; t < num_tuples; ++t) {
        s.len[t] = len[t];
        s.offset[t] = (uint32_t)total;
        for (uint32_t g = 0; g < 8; ++g)
            for (int j = 0; j < len[t]; ++j) s.src4[t][g][j] = (uint8_t)(4u * ntuple_sym_src(g, cells[kNTupleMaxLen * t + j]));
        total += (int64_t)1 << (4 * len[t]);
    }
    return total;
}

// every byte of x clamped to 15
#if defined(__CUDACC__)
ML2048_FN uint32_t min15_bytes(uint32_t x) { return __vminu4(x, 0x0f0f0f0fu); }
#else
ML2048_FN uint32_t min15_bytes(uint32_t x)
{
    uint32_t d = 0;
    for (int i = 0; i < 4; ++i) {
        const uint32_t b = (x >> (8 * i)) & 0xffu;
        d |= (b < 15u ? b : 15u) << (8 * i);
    }
    return d;
}
#endif

// The board as sixteen 4-bit fields, cell k (clamped to 15) in bits 4k..4k+3
ML2048_FN uint64_t ntuple_nibbles(uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3)
{
    const uint32_t w[4] = {r0, r1, r2, r3};
    uint64_t nib = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        uint32_t x = min15_bytes(w[i]);
        x = (x | (x >> 4)) & 0x00ff00ffu;  // bytes 0 and 2 hold two fields each
        x = (x | (x >> 8)) & 0xffffu;
        nib |= (uint64_t)x << (16 * i);
    }
    return nib;
}

// Table index of one tuple image: `src4` = its row of NTupleSpec::src4, `len` = the tuple's length
ML2048_FN uint32_t ntuple_index(uint64_t nib, const uint8_t *src4, uint32_t len)
{
    uint32_t idx = 0;
#pragma unroll
    for (uint32_t j = 0; j < (uint32_t)kNTupleMaxLen; ++j)
        if (j < len) idx |= (uint32_t)((nib >> src4[j]) & 15u) << (4u * j);
    return idx;
}

// Visit the 8K table entries of a board in the fixed order t = 0..K-1, g = 0..7: visit(offset, index) with offset = tuple
// t's first entry and index = image g's entry within that table, so entry j = offset + index of every weight-sized array.
template <class Visit>
ML2048_FN void ntuple_for_each_entry(const NTupleSpec &s, uint64_t nib, Visit &&visit)
{
    for (uint32_t t = 0; t < s.num_tuples; ++t) {
        const uint32_t off = s.offset[t], len = s.len[t];
#pragma unroll
        for (uint32_t g = 0; g < 8; ++g) visit(off, ntuple_index(nib, s.src4[t][g], len));
    }
}

#if defined(__CUDACC__)
ML2048_FN float load_weight(const float *p) { return __ldg(p); }
#else
ML2048_FN float load_weight(const float *p) { return *p; }
#endif

// ---- multi-stage n-tuple networks ----
// S (1..8) weight sets, one per stage of the game, given by S - 1 strictly ascending tile exponents tau_1 < ... < tau_{S-1} in
// 1..15.  m(b) = max over the 16 cells of min(b[c], 15) (the index's own clamp), stage(b) = #{k : tau_k <= m(b)}: an empty
// board is in stage 0, a byte >= 16 counts as 15.  The weights are S * N entries (N = sum_t 16^len_t), stage s's tables at
// s * N in the single-stage layout; every entry index s * N + offset_t + idx < 8 * 2^28 fits in 32 bits.  A board's value and
// every update use the tables of the board's own stage.  NTupleSpec itself stays the single-stage network (S = 1 runs the
// kernels' NTupleSpec instances); the staged spec extends it, so that the parameters of the existing kernels keep their offsets.
constexpr int kNTupleMaxStages = 8;

struct NTupleStagedSpec : NTupleSpec {
    uint32_t stage_size;  // N
    uint64_t stage_of;    // bits 4m..4m+3: the stage of a board whose largest clamped cell is m
};

// Host side: the stage table of validated thresholds (tau [S-1], ascending in 1..15)
inline uint64_t ntuple_stage_table(const uint8_t *tau, int32_t num_stages)
{
    uint64_t t = 0;
    for (uint32_t m = 0; m < 16u; ++m) {
        uint64_t s = 0;
        for (int k = 0; k + 1 < num_stages; ++k) s += tau[k] <= m ? 1u : 0u;
        t |= s << (4u * m);
    }
    return t;
}

// the largest of the 4 bytes of x, in byte 0
#if defined(__CUDACC__)
ML2048_FN uint32_t max_byte(uint32_t x)
{
    x = __vmaxu4(x, x >> 16);
    return __vmaxu4(x, x >> 8) & 0xffu;
}
ML2048_FN uint32_t max_bytes(uint32_t x, uint32_t y) { return __vmaxu4(x, y); }
#else
ML2048_FN uint32_t max_byte(uint32_t x)
{
    uint32_t m = 0;
    for (int i = 0; i < 4; ++i) m = ((x >> (8 * i)) & 0xffu) > m ? (x >> (8 * i)) & 0xffu : m;
    return m;
}
ML2048_FN uint32_t max_bytes(uint32_t x, uint32_t y)
{
    uint32_t d = 0;
    for (int i = 0; i < 4; ++i) {
        const uint32_t a = (x >> (8 * i)) & 0xffu, b = (y >> (8 * i)) & 0xffu;
        d |= (a > b ? a : b) << (8 * i);
    }
    return d;
}
#endif

// stage(b) from the board's clamped nibbles: the 16 fields split into two words of byte lanes, a byte-wise max, one shift of
// the stage table
ML2048_FN uint32_t ntuple_stage(const NTupleStagedSpec &s, uint64_t nib)
{
    const uint32_t lo = (uint32_t)nib, hi = (uint32_t)(nib >> 32);
    const uint32_t m = max_byte(max_bytes(max_bytes(lo & 0x0f0f0f0fu, (lo >> 4) & 0x0f0f0f0fu),
                                          max_bytes(hi & 0x0f0f0f0fu, (hi >> 4) & 0x0f0f0f0fu)));
    return (uint32_t)(s.stage_of >> (4u * m)) & 15u;
}

// The staged visitor: ntuple_for_each_entry over the tables of the board's stage (offset + stage(b) * N)
template <class Visit>
ML2048_FN void ntuple_for_each_entry(const NTupleStagedSpec &s, uint64_t nib, Visit &&visit)
{
    const uint32_t base = ntuple_stage(s, nib) * s.stage_size;
    ntuple_for_each_entry(static_cast<const NTupleSpec &>(s), nib, [&](uint32_t off, uint32_t idx) { visit(base + off, idx); });
}

// V(s): float32 adds from 0.0f in the fixed order t = 0..K-1, g = 0..7 -- bit-reproducible, and a sequential float32 reference
// matches it exactly.  Spec = NTupleSpec, or NTupleStagedSpec (the tables of the board's stage).
template <class Spec>
ML2048_FN float ntuple_value(const float *w, const Spec &s, uint64_t nib)
{
    float acc = 0.0f;
    ntuple_for_each_entry(s, nib, [&](uint32_t off, uint32_t idx) { acc += load_weight(w + off + idx); });
    return acc;
}

// ---- weight promotion of multi-stage networks (Jaskowski 2018) ----
// promoted: N bytes (N = sum_t 16^len_t, the single-stage entry count, for any S), indexed like a single-stage table.  Bit
// s - 1 of byte e is set once stage s's entry e has been written (s = 1..S-1); stage 0 has no mark, and bits S-1..7 are
// neither read nor written.  The effective weight is W(0, e) = w[e] and, for s >= 1, W(s, e) = w[s * N + e] if the mark of
// (s, e) is set, else W(s - 1, e): the source stage src(s, m) is the highest k <= s with k = 0 or bit k - 1 of m set.  Every
// read computes today's value, in the same float32 order, with W in place of w, so the storage of an unmarked entry is never
// read.  An update (ml2048_promoted_* in the header) first computes its deltas this way, then promotes: every masked-in game
// whose x_0 is in stage s0 >= 1 sets, for each of its entries e with (s0, e) unmarked, w[s0 * N + e] := W(s0 - 1, e) (TC:
// coherence {0, 0}) and the mark; then it applies the rule to x_0's own-stage entries as a staged update does.  So
// promotion changes no effective weight, and only the apply step does.
struct NTuplePromotedSpec : NTupleStagedSpec {
    const uint8_t *promoted;  // [N]
};

#if defined(__CUDACC__)
ML2048_FN uint32_t clz32(uint32_t x) { return (uint32_t)__clz(x); }
ML2048_FN uint32_t load_mark(const uint8_t *p) { return __ldg(p); }
#else
ML2048_FN uint32_t clz32(uint32_t x) { return (uint32_t)__builtin_clz(x); }
ML2048_FN uint32_t load_mark(const uint8_t *p) { return *p; }
#endif

// src(s, m) for a stage s in 0..7 and a mark byte m: bit 0 of the operand stands for stage 0, which is always written
ML2048_FN uint32_t ntuple_source_stage(uint32_t s, uint32_t m)
{
    return 31u - clz32(((m << 1) | 1u) & ((2u << s) - 1u));
}

// V(s) of a promoting network: each entry of the board's stage is read from its source stage.  A stage-0 board reads no mark.
ML2048_FN float ntuple_value(const float *w, const NTuplePromotedSpec &s, uint64_t nib)
{
    const uint32_t stage = ntuple_stage(s, nib);
    float acc = 0.0f;
    ntuple_for_each_entry(static_cast<const NTupleSpec &>(s), nib, [&](uint32_t off, uint32_t idx) {
        const uint32_t e = off + idx;
        const uint32_t src = stage ? ntuple_source_stage(stage, load_mark(s.promoted + e)) : 0u;
        acc += load_weight(w + src * s.stage_size + e);
    });
    return acc;
}

}  // namespace ml2048
