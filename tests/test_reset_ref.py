"""The NumPy references of the auto-reset bookkeeping (tests/_reset_ref.py) against brute-force Python loops (CPU)."""

from __future__ import annotations

import numpy as np
import pytest

import _reset_ref as ref


def _scan_brute(flags, group, chunk):
    counts = []
    for g in range(0, len(flags), group):
        counts.append(sum(int(x) for x in flags[g:g + group]))
    rank, bases, below_chunk, in_chunk = [], [], 0, 0
    for w, c in enumerate(counts):
        if w % chunk == 0:
            bases.append(below_chunk)
            in_chunk = 0
        rank.append(in_chunk)
        in_chunk += c
        below_chunk += c
    return counts, rank, bases, below_chunk


@pytest.mark.parametrize("group,chunk", [(32, 1024), (4, 3), (1, 1), (2, 5)])
@pytest.mark.parametrize("m", [1, 2, 5, 31, 32, 33, 97, 1000])
def test_scan_ref_equals_brute_force(group, chunk, m):
    rng = np.random.default_rng(m * 7 + group)
    for p in (0.0, 0.03, 0.5, 1.0):
        flags = (rng.random(m) < p).astype(np.uint8)
        got = ref.scan_ref(flags, group, chunk)
        counts, rank, bases, total = _scan_brute(flags, group, chunk)
        assert -(-m // group) == len(got.group_counts) == len(got.reset_rank)
        assert -(-len(counts) // chunk) == len(got.reset_chunk_base)
        np.testing.assert_array_equal(got.group_counts, counts)
        np.testing.assert_array_equal(got.reset_rank, rank)
        np.testing.assert_array_equal(got.reset_chunk_base, bases)
        assert got.total == total
        # the rank of a finished slot among all finished slots is chunk base + rank + finished slots before it in its group
        idx = np.flatnonzero(flags)
        w = idx // group
        order = got.reset_chunk_base[w // chunk] + got.reset_rank[w] + [int(flags[x - x % group:x].sum()) for x in idx]
        np.testing.assert_array_equal(order, np.arange(idx.size))


def test_scan_ref_refuses_non_binary_flags():
    with pytest.raises(AssertionError):
        ref.scan_ref(np.array([0, 2, 1], np.uint8))


@pytest.mark.parametrize("offset", [0, 5])
def test_prepare_ref_equals_brute_force(offset):
    flags = (np.random.default_rng(3).random(500) < 0.2).astype(np.uint8)
    got = ref.prepare_ref(flags, 1000, offset)
    want_idx = [i for i in range(500) if flags[i]]
    np.testing.assert_array_equal(got.indices, want_idx)
    np.testing.assert_array_equal(got.ids, [1000 + offset + k for k in range(len(want_idx))])
    assert got.n == len(want_idx) and got.game_count == 1000 + len(want_idx)


def test_flag_patterns():
    m = 1025 * ref.CHUNK_SLOTS + 9
    pats = {name: ref.flag_pattern(name, m, seed=1) for name in ref.PATTERNS}
    for name, f in pats.items():
        assert f.dtype == np.uint8 and f.shape == (m,) and f.max() <= 1, name
    assert pats["none"].sum() == 0 and pats["all"].sum() == m
    np.testing.assert_array_equal(np.flatnonzero(pats["first"]), [0])
    np.testing.assert_array_equal(np.flatnonzero(pats["last"]), [m - 1])
    for name, size in (("group", ref.GROUP), ("chunk", ref.CHUNK_SLOTS), ("tile", ref.TILE)):
        np.testing.assert_array_equal(np.flatnonzero(pats["last_of_" + name]), np.arange(size - 1, m, size))
    np.testing.assert_array_equal(np.flatnonzero(pats["first_of_chunk"]), np.arange(0, m, ref.CHUNK_SLOTS))
    np.testing.assert_array_equal(np.flatnonzero(pats["chunk1024"]), np.arange(1024 * ref.CHUNK_SLOTS, 1025 * ref.CHUNK_SLOTS))
    np.testing.assert_array_equal(np.flatnonzero(pats["tile1024"]), np.arange(1024 * ref.TILE, 1025 * ref.TILE))
    assert pats["alternating"].sum() == m // 2
    assert abs(pats["random1"].mean() - 0.01) < 0.001 and abs(pats["random50"].mean() - 0.5) < 0.001
    np.testing.assert_array_equal(pats["random1"], ref.flag_pattern("random1", m, seed=1))
    # the chunk-1024 pattern leaves the first pass of the scan without a reset: only the carry places its ranks
    s = ref.scan_ref(pats["chunk1024"])
    assert len(s.reset_chunk_base) == 1026 and s.reset_chunk_base[1024] == 0 and s.reset_chunk_base[1025] == ref.CHUNK_SLOTS
    assert ref.scan_ref(pats["first_of_chunk"]).reset_chunk_base[1024] == 1024


def test_dead_board_has_no_legal_move():
    b = ref.DEAD_BOARD.reshape(4, 4)
    assert (b > 0).all()
    assert not (b[:, 1:] == b[:, :-1]).any() and not (b[1:, :] == b[:-1, :]).any()
