"""
Expectimax without a GPU: the vectorised NumPy definition in tests/_expectimax_ref.py against a plain scalar recursion
written from the definition, both over the C oracle's moves and rewards; the C argument checks of ml2048_expectimax, which
return before any launch; and its header declaration compiled from C.
"""

from __future__ import annotations

import math
import os
import re
import subprocess

import numpy as np
import pytest

import _expectimax_ref as xref
import _ntuple_ref as ref

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(HERE), "include", "ml2048_b200.h")
KINDS = ("normal", "improved", "rank", "maxcell")
TWO_PROBS = (0.0, 0.3, 0.8, 1.0)


@pytest.fixture(scope="module")
def lib():
    from ml2048_b200 import _lib, build

    build.build()  # nvcc cross-compiles without a GPU; no-op when up to date
    return _lib.load()


# ---- the definition, one board at a time -------------------------------------------------------------


class Scalar:
    """E, M and the root straight from the definition, one float32 operation at a time"""

    def __init__(self, oracle, kind, w, tuples, two_prob):
        self.move = xref.oracle_move(oracle, kind)
        self.w, self.tuples = w, tuples
        self.p2 = np.float32(two_prob)
        self.p4 = np.float32(np.float32(1) - self.p2)

    def moves(self, b):
        after, reward, valid = self.move(b[None])
        return after[0], reward[0], valid[0]

    def V(self, s):
        return ref.value(s[None], self.w, self.tuples)[0]

    def M(self, b, d):
        after, reward, valid = self.moves(b)
        best = None
        for a in range(4):
            if not valid[a]:
                continue
            x = np.float32(reward[a] + (self.V(after[a]) if d == 1 else self.E(after[a], d - 1)))
            k = np.float32(-np.inf) if math.isnan(x) else x
            if best is None or k > best:
                best = k
        return np.float32(0) if best is None else best

    def E(self, s, d):
        cells = [c for c in range(16) if s[c] == 0]
        assert cells
        total = None
        for c in cells:
            t = None
            for tile, p in ((1, self.p2), (2, self.p4)):
                if p == 0:
                    continue
                child = s.copy()
                child[c] = tile
                term = np.float32(p * self.M(child, d))
                t = term if t is None else np.float32(t + term)
            total = t if total is None else np.float32(total + t)
        return np.float32(total / np.float32(len(cells)))

    def root(self, b, depth):
        after, reward, valid = self.moves(b)
        q = [np.float32(-np.inf)] * 4
        e = [np.float32(0)] * 4
        best = None
        for a in range(4):
            if valid[a]:
                e[a] = self.E(after[a], depth)
                q[a] = np.float32(reward[a] + e[a])
                k = np.float32(-np.inf) if math.isnan(q[a]) else q[a]
                if best is None or k > best[0]:
                    best = (k, a)
        if best is None:
            return 0, b, np.float32(0), np.float32(0), np.array(q, np.float32)
        a = best[1]
        return a, after[a], reward[a], e[a], np.array(q, np.float32)


def _same_bits(got, want):
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan)
    np.testing.assert_array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))


def _boards(rng, m: int, empties=(0, 15)) -> np.ndarray:
    """boards of exponents 1..15 with a number of empty cells drawn from `empties`, plus the edge cases"""
    b = rng.integers(1, 16, size=(m, 16)).astype(np.uint8)
    for i in range(m):
        k = int(rng.integers(empties[0], empties[1] + 1))
        b[i, rng.permutation(16)[:k]] = 0
    edge = [
        np.array([1, 2, 1, 2, 2, 1, 2, 1, 1, 2, 1, 2, 2, 1, 2, 1], np.uint8),    # dead: no valid move
        np.array([1, 0, 0, 0] + [0] * 12, np.uint8),                             # one tile: 15 empty cells after a move
        np.array([1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 0], np.uint8),  # one empty cell, moves leave one
        np.array([1, 2, 3, 4, 2, 3, 4, 5, 3, 4, 5, 6, 4, 5, 6, 6], np.uint8),    # full, one fusion: one empty after it
        np.array([1, 2, 3, 4, 5, 6, 7, 8, 1, 2, 3, 4, 5, 6, 7, 0], np.uint8),    # few valid moves
        np.array([15, 15, 14, 0, 13, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0], np.uint8),  # 15s that fuse
    ]
    return np.concatenate([np.stack(edge), b])


def _check(got: dict, want) -> None:
    a, st, r, v, q = want
    assert int(got["action"]) == a
    np.testing.assert_array_equal(got["state"], st)
    _same_bits(got["reward"], r)
    _same_bits(got["value"], v)
    _same_bits(got["q"], q)


@pytest.mark.parametrize("kind", KINDS)
def test_vectorised_reference_matches_scalar_depth1(oracle, kind):
    rng = np.random.default_rng(KINDS.index(kind))
    tuples = ((0, 1, 2, 3), (4, 5, 6, 7), (0, 4, 8, 12), (1, 5))
    w = (rng.standard_normal(ref.num_weights(tuples)) * 50).astype(np.float32)
    w[rng.random(w.size) < 0.3] = 0.0  # zero entries: ties and signed zeros
    boards = _boards(rng, 100)
    for two_prob in TWO_PROBS:
        got = xref.expectimax(boards, w, tuples, depth=1, two_prob=two_prob, move=xref.oracle_move(oracle, kind))
        sc = Scalar(oracle, kind, w, tuples, two_prob)
        for i in range(boards.shape[0]) if two_prob == 0.8 else rng.integers(0, boards.shape[0], 20):
            _check({k: v[i] for k, v in got.items()}, sc.root(boards[i], 1))
    assert got["action"][0] == 0 and (got["q"][0] == -np.inf).all() and got["value"][0] == 0  # the dead board


@pytest.mark.parametrize("kind", KINDS)
def test_vectorised_reference_matches_scalar_depth2(oracle, kind):
    rng = np.random.default_rng(10 + KINDS.index(kind))
    tuples = ((0, 1, 2), (5, 6, 9, 10))
    w = (rng.standard_normal(ref.num_weights(tuples)) * 50).astype(np.float32)
    boards = _boards(rng, 24, empties=(0, 3))
    boards = np.concatenate([boards[[0, 2, 3, 4]], boards[6:]])  # the edge boards with few empty cells
    two_prob = TWO_PROBS[KINDS.index(kind)]
    got = xref.expectimax(boards, w, tuples, depth=2, two_prob=two_prob, move=xref.oracle_move(oracle, kind))
    sc = Scalar(oracle, kind, w, tuples, two_prob)
    for i in range(boards.shape[0]):
        _check({k: v[i] for k, v in got.items()}, sc.root(boards[i], 2))


def test_vectorised_reference_nan_inf_and_zero_weights(oracle):
    rng = np.random.default_rng(20)
    tuples = ((0, 1, 2, 3), (3, 7, 11))
    n = ref.num_weights(tuples)
    boards = _boards(rng, 40)
    for w in (np.zeros(n, np.float32), np.where(rng.random(n) < 0.2, np.nan, rng.standard_normal(n)).astype(np.float32),
              np.where(rng.random(n) < 0.1, -np.inf, np.where(rng.random(n) < 0.05, np.inf, rng.standard_normal(n))).astype(np.float32)):
        got = xref.expectimax(boards, w, tuples, depth=1, two_prob=0.3, move=xref.oracle_move(oracle, "rank"))
        sc = Scalar(oracle, "rank", w, tuples, 0.3)
        for i in range(boards.shape[0]):
            _check({k: v[i] for k, v in got.items()}, sc.root(boards[i], 1))


def test_two_prob_extremes_use_one_tile():
    """two_prob = 1 never evaluates a 4, two_prob = 0 never a 2: a move function that sees only the other tile fails"""
    seen = set()

    def move(boards):
        seen.update(int(x) for x in np.unique(boards))
        m = boards.shape[0]
        after = np.repeat(boards[:, None], 4, axis=1)
        after[:, :, 15] = 0  # a "move" that clears cell 15 of a full board
        valid = np.zeros((m, 4), bool)
        valid[:, 0] = boards[:, 15] != 0
        return after, np.zeros((m, 4), np.float32), valid

    b = np.zeros((1, 16), np.uint8)
    b[0, :] = 3
    for two_prob, tile in ((1.0, 1), (0.0, 2)):
        seen.clear()
        xref.expectimax(b, np.zeros(16, np.float32), ((0,),), depth=2, two_prob=two_prob, move=move)
        assert tile in seen and (3 - tile) not in seen


# ---- the C arguments -------------------------------------------------------------------------------------


def test_c_argument_errors_without_gpu(lib):
    """every check returns before a launch (the pointers below are never dereferenced)"""
    cells = np.zeros((2, 6), np.uint8)
    cells[0, :2] = (0, 1)
    cells[1, 0] = 5
    lens = np.array([2, 1], np.uint8)
    n = 16 ** 2 + 16
    B, W, O = 0x10000, 0x20000, 0x30000

    def call(*, board=B, w=W, nw=n, cl=cells.ctypes.data, ln=lens.ctypes.data, k=2, kind=0, depth=1, p=0.8, u8=O, i64=None,
             after=0x40000, reward=0x50000, value=0x60000, q=0x70000, m=8):
        return lib.ml2048_expectimax(board, w, nw, cl, ln, k, kind, depth, p, u8, i64, after, reward, value, q, m, None)

    assert call(m=0) == -3 and call(m=-1) == -3
    for arg in ("board", "w", "after", "reward", "value", "q", "cl", "ln"):
        assert call(**{arg: None}) == -1, arg
    assert call(u8=None) == -1
    assert call(board=B + 4) == -2 and call(w=W + 2) == -2 and call(u8=None, i64=O + 4) == -2
    assert call(after=0x40008) == -2 and call(reward=0x50002) == -2 and call(value=0x60001) == -2 and call(q=0x70002) == -2
    assert call(kind=4) == -4 and call(kind=-1) == -4
    for depth in (0, 3, -1):
        assert call(depth=depth) == -4
    for p in (-0.01, 1.01, float("nan"), float("inf"), -float("inf")):
        assert call(p=p) == -4, p
    assert call(k=0) == -3 and call(k=17) == -3 and call(nw=n + 1) == -3
    bad = cells.copy()
    bad[0, 1] = 0  # a repeated cell
    assert call(cl=bad.ctypes.data) == -4


def test_python_argument_errors_without_gpu():
    import torch

    from ml2048_b200 import ops
    from ml2048_b200.ntuple import ExpectimaxPolicy

    b = torch.zeros((4, 16), dtype=torch.uint8)
    w = torch.zeros(16, dtype=torch.float32)
    with pytest.raises(ValueError):
        ops.ntuple_expectimax(b, w, [[0]])  # CPU tensors
    with pytest.raises(ValueError):
        ops.ntuple_expectimax(torch.zeros((4, 15), dtype=torch.uint8), w, [[0]])
    for bad in ({"depth": 0}, {"depth": 3}, {"depth": True}, {"two_prob": 1.5}, {"two_prob": float("nan")}, {"two_prob": "x"},
                {"action_dtype": torch.int32}, {"reward_fn": lambda s, p, m: 0.0}):
        with pytest.raises(ValueError):
            ops.ntuple_expectimax(b, w, [[0]], **bad)
    with pytest.raises(ValueError):
        ExpectimaxPolicy(None, depth=3)


def test_header_declaration_compiles(tmp_path):
    """ml2048_expectimax compiles from C with its documented argument types, and _lib.SYMBOLS binds it"""
    from ml2048_b200 import _lib

    src = tmp_path / "xm.c"
    src.write_text(
        f'#include "{HEADER}"\n'
        "int f(void *b, float *w, uint8_t *c, uint8_t *l, float *v, uint8_t *a8, int64_t *a64, void *s) {\n"
        "  return ml2048_expectimax(b, w, 16, c, l, 1, 0, 2, 0.9, a8, a64, b, v, v, v, 1, s);\n}\n")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-c", str(src), "-o", str(tmp_path / "xm.o")], check=True)
    assert re.search(r"ML2048_API\s+int\s+ml2048_expectimax\s*\(", open(HEADER).read())
    assert "ml2048_expectimax" in _lib.SYMBOLS
    assert _lib.ABI_VERSION == 12
