"""
The product's device arithmetic (ml2048_b200/csrc/board_ops.cuh) compiled as plain C++ (tests/host_shim)
and checked against the CPU oracle / golden fixtures WITHOUT a GPU: every 4-cell line in every board
position and direction (18^4 x 4 x 4), the reference-generated board set, random boards for the mask,
the replay spawn position, and Philox against its published known-answer vectors.  The masked categorical sampler is
checked against the float64 reference of tests/_rollout_ref.py.
"""

from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import golden

HERE = os.path.dirname(os.path.abspath(__file__))
SHIM_SRC = os.path.join(HERE, "host_shim", "board_ops_host.cpp")
SHIM_LIB = os.path.join(HERE, "host_shim", "libboard_ops_host.so")
HEADER = os.path.join(os.path.dirname(HERE), "ml2048_b200", "csrc", "board_ops.cuh")


@pytest.fixture(scope="module")
def shim():
    if not os.path.exists(SHIM_LIB) or os.path.getmtime(SHIM_LIB) < max(os.path.getmtime(SHIM_SRC), os.path.getmtime(HEADER)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", SHIM_LIB, SHIM_SRC],
                       check=True)
    lib = ctypes.CDLL(SHIM_LIB)
    vp, i64, u32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_uint32
    lib.hs_move_batch.argtypes = [vp, i64, ctypes.c_int, vp, vp, vp, vp, vp, vp]
    lib.hs_first_empty_batch.argtypes = [vp, vp, i64, vp]
    lib.hs_valid_mask.argtypes = [vp]
    lib.hs_valid_mask.restype = u32
    lib.hs_max_cell.argtypes = [vp]
    lib.hs_max_cell.restype = u32
    lib.hs_empties16.argtypes = [vp]
    lib.hs_empties16.restype = u32
    lib.hs_kth_set_bit16.argtypes = [u32, u32]
    lib.hs_kth_set_bit16.restype = u32
    lib.hs_philox.argtypes = [vp, vp, vp]
    lib.hs_philox2.argtypes = [vp, u32, vp]
    lib.hs_slot_draws.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, u32, vp]
    lib.hs_slot_word.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, u32]
    lib.hs_slot_word.restype = u32
    lib.hs_sample_masked_categorical_batch.argtypes = [vp, vp, vp, i64, vp, vp]
    return lib


def _move_batch(shim, boards, action):
    n = boards.shape[0]
    b = np.ascontiguousarray(boards, np.uint8)
    out = np.empty_like(b)
    gain = np.empty(n, np.uint32)
    rank = np.empty(n, np.uint32)
    count = np.empty(n, np.uint32)
    merged = np.empty((n, 16), np.uint8)
    mask = np.empty(n, np.uint32)
    shim.hs_move_batch(b.ctypes.data, n, action, out.ctypes.data, gain.ctypes.data, rank.ctypes.data, count.ctypes.data,
                       merged.ctypes.data, mask.ctypes.data)
    return out, gain, rank, count, merged, mask.view(np.uint8).reshape(n, 4)


def test_every_line_every_position_every_direction(shim):
    """All 18^4 lines, as each of the 4 rows (left/right) and each of the 4 columns (up/down), with noise
    in the other cells, against the reference's own _push_row table (tests/golden/line_table.npz)."""
    tab = golden("line_table.npz")
    v = np.arange(18, dtype=np.uint8)
    lines = np.stack(np.meshgrid(v, v, v, v, indexing="ij"), axis=-1).reshape(-1, 4)
    n = lines.shape[0]
    rng = np.random.default_rng(1)
    weights = (2 << np.arange(18)).astype(np.int64)
    for action, name in ((0, "first"), (1, "last"), (2, "first"), (3, "last")):
        pushed, fused = tab[f"pushed_{name}"], tab[f"fused_{name}"]
        want_gain = np.where(fused > 0, weights[fused], 0).sum(axis=1)
        for pos in range(4):
            boards = rng.integers(0, 18, size=(n, 16)).astype(np.uint8).reshape(n, 4, 4)
            if action < 2:
                boards[:, pos, :] = lines
            else:
                boards[:, :, pos] = lines
            out, gain, rank, count, merged, _ = _move_batch(shim, boards.reshape(n, 16), action)
            out = out.reshape(n, 4, 4)
            got = out[:, pos, :] if action < 2 else out[:, :, pos]
            bad = np.flatnonzero((got != pushed).any(axis=1))
            assert bad.size == 0, (action, pos, lines[bad[0]], got[bad[0]], pushed[bad[0]])
        # rewards / merged on boards where only this line can fuse (other lines all distinct, no zeros needed)
        filler = np.array([[1, 2, 3, 4], [5, 6, 7, 8], [9, 10, 11, 12], [13, 14, 15, 16]], np.uint8)
        boards = np.broadcast_to(filler if action < 2 else filler.T, (n, 4, 4)).copy()
        if action < 2:
            boards[:, 0, :] = lines
        else:
            boards[:, :, 0] = lines
        out, gain, rank, count, merged, _ = _move_batch(shim, boards.reshape(n, 16), action)
        np.testing.assert_array_equal(gain.astype(np.int64), want_gain)
        np.testing.assert_array_equal(count, (fused > 0).sum(axis=1))
        np.testing.assert_array_equal(rank, np.where(fused > 0, fused.astype(np.int64) + 1, 0).sum(axis=1))
        want_merged = np.zeros((n, 18), np.uint8)
        for j in range(2):
            np.add.at(want_merged, (np.arange(n), fused[:, j]), (fused[:, j] > 0).astype(np.uint8))
        np.testing.assert_array_equal(merged, want_merged[:, :16])


def test_reference_board_set(shim, oracle):
    g = golden("boards.npz")
    boards = g["boards"]
    names = [str(x) for x in g["reward_names"]]
    for action in range(4):
        out, gain, rank, count, merged, mask = _move_batch(shim, boards, action)
        np.testing.assert_array_equal(out, g["moved"][:, action])
        np.testing.assert_array_equal(merged, g["merged"][:, action])
        np.testing.assert_array_equal(mask, g["mask"])
        np.testing.assert_array_equal(gain.astype(np.float64), g["rewards"][:, action, names.index("normal")])
        np.testing.assert_array_equal(rank.astype(np.float64), g["rewards"][:, action, names.index("rank")])
        # "the move changes the board" == valid_actions[action] (game_numba.py:718)
        np.testing.assert_array_equal((out != boards).any(axis=1), g["mask"][:, action] != 0)


def test_mask_and_max_on_random_boards(shim, oracle):
    rng = np.random.default_rng(5)
    n = 20000
    dens = rng.choice([0.1, 0.5, 0.9, 1.0], size=n)
    hi = rng.choice([2, 3, 5, 17], size=n)
    boards = (rng.integers(0, 1 << 30, size=(n, 16)) % hi[:, None] + 1).astype(np.uint8)
    boards[rng.random((n, 16)) >= dens[:, None]] = 0
    for i in range(n):
        got = shim.hs_valid_mask(boards[i].ctypes.data)
        want = int(oracle.board_valid(boards[i]).view(np.uint32)[0])
        assert got == want, (boards[i], hex(got), hex(want))
        assert shim.hs_max_cell(boards[i].ctypes.data) == boards[i].max()
        e = shim.hs_empties16(boards[i].ctypes.data)
        assert e == sum(1 << c for c in range(16) if boards[i][c] == 0)


def test_spawn_position_matches_table_walk(shim):
    """first_empty_by_rank on the inverse-form keys == the reference's walk over the permutation row."""
    rng = np.random.default_rng(9)
    n = 50000
    perms = np.argsort(rng.random((n, 16)), axis=1).astype(np.uint8)
    keys = np.empty((n, 16), np.uint8)
    keys[np.arange(n)[:, None], perms] = (np.arange(16, dtype=np.uint8) * 16)[None, :] + perms
    boards = rng.integers(1, 5, size=(n, 16)).astype(np.uint8)
    boards[rng.random((n, 16)) < rng.random((n, 1))] = 0
    boards[:50] = 1  # full boards
    boards[50:100] = 1
    boards[50:100, 15] = 0  # only cell 15 empty (its key can be 0xff)
    cells = np.empty(n, np.uint32)
    shim.hs_first_empty_batch(keys.ctypes.data, boards.ctypes.data, n, cells.ctypes.data)
    empty_in_order = np.take_along_axis(boards, perms.astype(np.int64), axis=1) == 0
    want = np.where(empty_in_order.any(axis=1), perms[np.arange(n), empty_in_order.argmax(axis=1)], 16)
    np.testing.assert_array_equal(cells, want)


def test_kth_set_bit(shim):
    for mask in list(range(1, 1 << 12, 37)) + [0xFFFF, 0x8000, 0x0001, 0xF0F0]:
        bits = [i for i in range(16) if mask >> i & 1]
        for k, want in enumerate(bits):
            assert shim.hs_kth_set_bit16(mask, k) == want


def test_action_mask_helpers(shim):
    shim.hs_mask_bits4.restype = ctypes.c_uint32
    shim.hs_kth_valid_action.restype = ctypes.c_uint32
    for bits in range(16):
        word = sum(1 << (8 * i) for i in range(4) if bits >> i & 1)
        assert shim.hs_mask_bits4(word) == bits
        valid = [i for i in range(4) if bits >> i & 1]
        for k, want in enumerate(valid):
            assert shim.hs_kth_valid_action(bits, k) == want


def test_philox_known_answers(shim):
    # Random123 kat_vectors: philox4x32-10
    cases = [
        ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
        ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
        ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
    ]
    for ctr, key, want in cases:
        c = np.array(ctr, np.uint32)
        k = np.array(key, np.uint32)
        out = np.zeros(4, np.uint32)
        shim.hs_philox(c.ctypes.data, k.ctypes.data, out.ctypes.data)
        assert tuple(int(x) for x in out) == want


def test_policy_selector_table(shim):
    """Row 4*bits + k of the random policy's table = the selector row of the k-th valid direction of `bits`, which it also
    names in word 6; rows 60..63 are the four directions in order."""
    shim.hs_policy_sel_table.argtypes = [ctypes.c_void_p]
    shim.hs_move_sel_table.argtypes = [ctypes.c_void_p]
    tab = np.zeros((64, 8), np.uint32)
    base = np.zeros((4, 8), np.uint32)
    shim.hs_policy_sel_table(tab.ctypes.data)
    shim.hs_move_sel_table(base.ctypes.data)
    for bits in range(16):
        valid = [d for d in range(4) if bits >> d & 1]
        for k in range(4):
            action = valid[k] if k < len(valid) else 0
            if k < len(valid):
                assert shim.hs_kth_valid_action(bits, k) == action
            row = tab[4 * bits + k]
            assert row[6] == action and row[7] == 0
            np.testing.assert_array_equal(row[:6], base[action][:6])
    assert [int(tab[60 + a][6]) for a in range(4)] == [0, 1, 2, 3]


def test_fresh_board_table(shim, oracle):
    """Every entry of the reset's lookup table = the two tiles placed with put_cell and the product's (and the oracle's)
    valid-action mask of that board."""
    shim.hs_fresh_table.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    shim.hs_put_cell.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32]
    boards = np.zeros((1024, 16), np.uint8)
    masks = np.zeros((1024,), np.uint32)
    shim.hs_fresh_table(boards.ctypes.data, masks.ctypes.data)
    for idx in range(1024):
        c0, c1, t0, t1 = idx >> 6, (idx >> 2) & 15, (idx >> 1) & 1, idx & 1
        b = np.zeros(16, np.uint8)
        shim.hs_put_cell(b.ctypes.data, c0, 2 - t0)
        shim.hs_put_cell(b.ctypes.data, c1, 2 - t1)
        np.testing.assert_array_equal(boards[idx], b)
        assert int(masks[idx]) == shim.hs_valid_mask(b.ctypes.data), idx
        if c0 != c1:
            assert masks[idx : idx + 1].view(np.uint8).tolist() == oracle.board_valid(b).tolist(), idx


PHILOX2X32_KAT = [  # Random123 kat_vectors: philox2x32 10
    ((0, 0), 0, (0xFF1DAE59, 0x6CD10DF2)),
    ((0xFFFFFFFF, 0xFFFFFFFF), 0xFFFFFFFF, (0x2C3F628B, 0xAB4FD7AD)),
    ((0x243F6A88, 0x85A308D3), 0x13198A2E, (0xDD7CE038, 0xF62A4C12)),
]


def test_philox2x32_known_answers(shim):
    """The block the kernels draw per game-step (board_ops.cuh:philox2x32_10), compiled for the host."""
    for ctr, key, want in PHILOX2X32_KAT:
        c = np.array(ctr, np.uint32)
        out = np.zeros(2, np.uint32)
        shim.hs_philox2(c.ctypes.data, key, out.ctypes.data)
        assert tuple(int(x) for x in out) == want


def test_slot_draws_key_schedule(shim):
    """slot_draws = Philox2x32-10 with counter (slot low, counter low ^ high words * odd constants) and key = seed ^ stream tag
    (uniform over a launch)."""
    def ref(slot, counter, seed, tag):
        m = 0xFFFFFFFF
        key = (seed & m) ^ (((seed >> 32) * 0x9E3779B9) & m) ^ tag
        c = np.array([slot & m, (counter & m) ^ (((counter >> 32) * 0x85EBCA6B) & m) ^ (((slot >> 32) * 0xC2B2AE35) & m)], np.uint32)
        out = np.zeros(2, np.uint32)
        shim.hs_philox2(c.ctypes.data, key, out.ctypes.data)
        return tuple(int(x) for x in out)

    out = np.zeros(2, np.uint32)
    seen = set()
    for slot, counter, seed, tag in ((0, 0, 0, 0), (5, 9, 123, 0), (5, 9, 123, 0x80000000), ((1 << 33) + 5, 9, 123, 0),
                                     (5, (1 << 40) + 9, 123, 0), (5, 9, (7 << 32) + 123, 0), ((1 << 27) - 1, 2**32 - 1, 2**64 - 1, 0)):
        shim.hs_slot_draws(slot, counter, seed, tag, out.ctypes.data)
        got = tuple(int(x) for x in out)
        assert got == ref(slot, counter, seed, tag)
        seen.add(got)
    assert len(seen) == 7  # high words and the stream tag all matter


def test_slot_word_serves_slot_pairs(shim):
    """slot_word: the policy / spawn word of a global slot is one half of the Philox block of its slot PAIR (index = slot >> 1;
    even slot -> .x, odd slot -> .y), for every stream tag."""
    out = np.zeros(2, np.uint32)
    for slot in (0, 1, 2, 3, 1000, 1001, (1 << 33) + 4, (1 << 33) + 5, 2**40 - 1):
        for counter, seed, tag in ((0, 0, 0), (77, 123, 0), (77, 123, 0x40000000), ((3 << 32) + 1, (9 << 32) + 4, 0)):
            shim.hs_slot_draws(slot >> 1, counter, seed, tag, out.ctypes.data)
            assert shim.hs_slot_word(slot, counter, seed, tag) == int(out[slot & 1])


def test_policy_words_reference(shim):
    """The tests' NumPy policy words (_rollout_ref.policy_words) == slot_word of the header and == the slot-pair formula over
    the library's host Philox2x32-10, for slot bases odd and beyond 2^32, counters and seeds beyond 2^32."""
    from _rollout_ref import policy_words

    from ml2048_b200 import _lib, build

    build.build()  # nvcc cross-compiles without a GPU; no-op when up to date
    lib = _lib.load()
    out2 = np.zeros(2, np.uint32)
    for base, counter, seed in ((0, 0, 0), (5001, 77, 123), ((1 << 34) + 17, (3 << 32) + 1, (9 << 32) + 4),
                                ((1 << 33) + 1, 2**64 - 1, 2**64 - 1)):
        slots = base + np.arange(64, dtype=np.uint64)
        got = policy_words(slots, counter, seed)
        for s, word in zip(slots.tolist(), got.tolist()):
            assert word == shim.hs_slot_word(s, counter, seed, 0), (s, counter, seed)
            key = (seed & 0xFFFFFFFF) ^ (((seed >> 32) * 0x9E3779B9) & 0xFFFFFFFF)
            pair = s >> 1
            c = np.array([pair & 0xFFFFFFFF, (counter & 0xFFFFFFFF) ^ (((counter >> 32) * 0x85EBCA6B) & 0xFFFFFFFF)
                          ^ (((pair >> 32) * 0xC2B2AE35) & 0xFFFFFFFF)], np.uint32)
            lib.ml2048_philox2x32_10(c.ctypes.data, key, out2.ctypes.data)
            assert word == int(out2[s & 1]), (s, counter, seed)


def _host_sampler(shim, words):
    def sample(logits, valid):
        n = logits.shape[0]
        bits = ((valid != 0) * (1 << np.arange(4))).sum(axis=1).astype(np.uint8)
        actions = np.empty(n, np.uint8)
        log_probs = np.empty(n, np.float32)
        shim.hs_sample_masked_categorical_batch(np.ascontiguousarray(logits, np.float32).ctypes.data, bits.ctypes.data,
                                                words.ctypes.data, n, actions.ctypes.data, log_probs.ctypes.data)
        return actions, log_probs

    return sample


def test_masked_categorical_sampler_against_float64(shim):
    """sample_masked_categorical compiled for the host, per logit class (randn*3, one dominant logit 80-120 above the rest,
    +-1e4, +-1e30, ties, and u placed on a CDF boundary) over all 16 masks with valid bytes 1..255: the inverse-CDF action
    of the float64 reference (either neighbour within 4*2^-24 of a boundary) and its log_softmax within
    2^-22 (|l_a| + |max logit|) + 2^-21."""
    import _rollout_ref as ref

    rng = np.random.default_rng(2024)
    n = 1 << 16
    words = ref.policy_words((1 << 34) + 17 + np.arange(n, dtype=np.uint64), (3 << 32) + 1, 0x9E3779B97F4A7C15)
    sample = _host_sampler(shim, words)
    seen = {}
    for name in ref.LOGIT_CLASSES:
        logits = ref.sampler_logits(name, rng, words)
        valid = ref.random_masks(rng, n)
        if name == "boundary":
            valid = ref.boundary_valid(valid)
        actions, log_probs = sample(logits, valid)
        seen[name] = ref.check_sampler(logits, valid, words, actions, log_probs, adversarial=name == "boundary", what=name)
    assert seen["boundary"]["boundary_rows"] > n // 4  # the adversarial class does reach the neighbour rule


def test_masked_categorical_sampler_exact_cases(shim):
    """One valid / no valid action, equal logits (including uniforms on the 1/3 and 2/3 boundaries), NaN / +-inf logits
    masked or valid: exact outcomes (_rollout_ref.check_sampler_exact)."""
    import _rollout_ref as ref

    words = ref.policy_words(5001 + np.arange(4099, dtype=np.uint64), 77, 123)
    words[:8] = (np.array([0x555555, 0x555556, 0xAAAAAA, 0xAAAAAB] * 2, np.uint32) << 8) | np.arange(8, dtype=np.uint32) * 31
    ref.check_sampler_exact(_host_sampler(shim, words), words, np.random.default_rng(7))


def test_hypothesis_boards_against_oracle(shim, oracle):
    """Property-based: arbitrary boards (exponents 0..17, any density) x any direction: the product's SWAR move, mask,
    max tile and fusion bookkeeping equal the oracle's scalar restatement of the reference."""
    from hypothesis import given, settings
    from hypothesis import strategies as st

    cells = st.lists(st.integers(min_value=0, max_value=17), min_size=16, max_size=16)

    @settings(max_examples=3000, deadline=None)
    @given(cells=cells, action=st.integers(min_value=0, max_value=3))
    def check(cells, action):
        board = np.array(cells, np.uint8)
        out, gain, rank, count, merged, mask = _move_batch(shim, board[None, :], action)
        want_board, want_merged18 = None, None
        b = board.copy()
        buckets = np.zeros(18, np.int64)
        # oracle line by line (its single-board entry point only has 16 merged slots, as the reference)
        lines = {0: [(4 * r, 1) for r in range(4)], 1: [(4 * r + 3, -1) for r in range(4)],
                 2: [(c, 4) for c in range(4)], 3: [(12 + c, -4) for c in range(4)]}[action]
        for first, stride in lines:
            idx = [first + k * stride for k in range(4)]
            pushed, bk = oracle.line_push(b[idx], False)
            b[idx] = pushed
            buckets += bk
        np.testing.assert_array_equal(out[0], b)
        assert int(gain[0]) == int(sum(int(buckets[k]) << (k + 1) for k in range(18)))
        assert int(count[0]) == int(buckets.sum())
        assert int(rank[0]) == int(sum((k + 1) * int(buckets[k]) for k in range(18)))
        np.testing.assert_array_equal(merged[0], buckets[:16].astype(np.uint8))
        np.testing.assert_array_equal(mask[0], oracle.board_valid(board))
        assert shim.hs_max_cell(board.ctypes.data) == board.max()

    check()
