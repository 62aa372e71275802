"""Plain NumPy references of the auto-reset's integer bookkeeping, shared by tests/test_reset_ref.py (CPU) and
tests/test_reset_bookkeeping.py (GPU):

    scan_ref      what ml2048_autoreset_scan computes from the `terminated` flags: finished games per group of 32 slots,
                  their exclusive prefix inside each chunk of 1024 groups (reset_rank), the exclusive prefix over the chunk
                  totals (reset_chunk_base) and the total
    prepare_ref   what one prepare() hands out: the reset slots (np.flatnonzero, game_numba.py:629), their ids (slot-ordered,
                  :641-644) and the next value of the id counter
    flag_pattern  seeded `terminated` patterns, among them ones that put every reset behind the first 1024 chunks or tiles
    DEAD_BOARD    a full board without a legal move
"""

from __future__ import annotations

from types import SimpleNamespace

import numpy as np

GROUP = 32                # slots per group of the auto-reset scan (one thread)
CHUNK = 1024              # groups per chunk (one block of the scan)
CHUNK_SLOTS = GROUP * CHUNK
TILE = 4096               # slots per tile of the three-launch prepare (count, scan, apply)
INT32_MAX = (1 << 31) - 1

# exponents 1 2 1 2 / 2 1 2 1 / ...: no empty cell and no two equal neighbours, so no move is legal
DEAD_BOARD = np.array([1, 2, 1, 2, 2, 1, 2, 1, 1, 2, 1, 2, 2, 1, 2, 1], dtype=np.uint8)

PATTERNS = ("none", "all", "first", "last", "last_of_group", "last_of_chunk", "last_of_tile", "first_of_chunk",
            "first_of_tile", "chunk1024", "tile1024", "alternating", "random1", "random50")


def _exclusive_cumsum(x: np.ndarray, axis: int = -1) -> np.ndarray:
    return np.cumsum(x, axis=axis, dtype=np.int64) - x


def scan_ref(flags, group: int = GROUP, chunk: int = CHUNK) -> SimpleNamespace:
    """The auto-reset scan of a 0/1 flag vector of length M, in int64: ``group_counts`` (finished games per group of
    `group` slots), ``reset_rank`` (for every group, the finished games in the lower groups of its chunk of `chunk`
    groups), ``reset_chunk_base`` (for every chunk, the finished games in the lower chunks) and ``total``."""
    f = np.asarray(flags)
    assert f.dtype == np.uint8 and f.ndim == 1 and f.size > 0 and f.max() <= 1, "flags are 0/1 bytes"
    m = f.size
    groups = -(-m // group)
    chunks = -(-groups // chunk)
    padded = np.zeros(groups * group, np.uint8)
    padded[:m] = f
    group_counts = padded.reshape(groups, group).sum(axis=1, dtype=np.int64)
    per_chunk = np.zeros(chunks * chunk, np.int64)
    per_chunk[:groups] = group_counts
    per_chunk = per_chunk.reshape(chunks, chunk)
    reset_rank = _exclusive_cumsum(per_chunk, axis=1).reshape(-1)[:groups]
    totals = per_chunk.sum(axis=1)
    reset_chunk_base = _exclusive_cumsum(totals)
    total = int(totals.sum())
    assert total == np.count_nonzero(f)
    for a in (group_counts, reset_rank, reset_chunk_base):
        assert a.min() >= 0 and a.max() <= INT32_MAX  # the kernel stores int32
    assert total <= INT32_MAX
    return SimpleNamespace(group_counts=group_counts, reset_rank=reset_rank, reset_chunk_base=reset_chunk_base, total=total)


def prepare_ref(flags, game_count: int, id_offset: int = 0) -> SimpleNamespace:
    """One prepare() of an unsharded batch from the id counter `game_count`: ``indices`` (the reset slots, ascending),
    ``ids`` (the ids they receive: game_count + id_offset + their rank) and ``game_count`` (the counter afterwards,
    advanced by the number of resets)."""
    indices = np.flatnonzero(np.asarray(flags))
    n = indices.size
    ids = int(game_count) + int(id_offset) + np.arange(n, dtype=np.int64)
    return SimpleNamespace(indices=indices, ids=ids, n=n, game_count=int(game_count) + n)


def flag_pattern(name: str, m: int, seed: int = 0) -> np.ndarray:
    """A uint8 0/1 `terminated` vector of length m.  The ``*1024`` patterns set every slot of chunk 1024 (the first chunk
    the second pass of the scan covers) or tile 1024 and nothing else; below that size they are empty."""
    f = np.zeros(m, np.uint8)
    if name == "none":
        pass
    elif name == "all":
        f[:] = 1
    elif name == "first":
        f[0] = 1
    elif name == "last":
        f[m - 1] = 1
    elif name.startswith("last_of_"):
        step = {"group": GROUP, "chunk": CHUNK_SLOTS, "tile": TILE}[name[len("last_of_"):]]
        f[step - 1::step] = 1
    elif name.startswith("first_of_"):
        step = {"chunk": CHUNK_SLOTS, "tile": TILE}[name[len("first_of_"):]]
        f[::step] = 1
    elif name in ("chunk1024", "tile1024"):
        size = CHUNK_SLOTS if name == "chunk1024" else TILE
        f[1024 * size:1025 * size] = 1
    elif name == "alternating":
        f[1::2] = 1
    elif name in ("random1", "random50"):
        p = 0.01 if name == "random1" else 0.5
        f[:] = np.random.default_rng(seed).random(m, dtype=np.float32) < p
    else:
        raise ValueError(name)
    return f
