"""Plain NumPy definition of ops.ntuple_expectimax, for the tests.

``move(boards)`` gives, for (N,16) uint8 boards, (after (N,4,16) uint8, reward (N,4) float32, valid (N,4)) exactly as
``ops.afterstates(boards, reward_fn=...)`` does; the GPU tests pass that op, the CPU tests a wrapper over the C oracle.  V is
``_ntuple_ref.value``.  p2 = float32(two_prob), p4 = float32(1) - p2.  Every operation is one float32 operation:

    E(s, d)  for the empty cells c_1 < ... < c_n of afterstate s: t_c = p2 * M(s + exponent 1 at c, d) + p4 * M(s + exponent 2
             at c, d) (p2 * m2 alone when p4 == 0, p4 * m4 alone when p2 == 0: an outcome of probability 0 is not evaluated);
             S = t_c1, then + t_c2, ... in ascending cell order; E = S / float(n)
    M(b, d)  max over the valid a of key(r(b,a) + (V(after(b,a)) if d == 1 else E(after(b,a), d - 1))), key(NaN) = -inf; among
             equal keys the smallest direction's key; 0 for a board without a valid move
    root     q_a = r(b,a) + E(after(b,a), D) for a valid a, -inf otherwise; the action is the argmax of key(q_a) with ties to the
             smallest direction; value = E(after(b,a*), D); a board without a valid move gets action 0, its own board,
             reward 0, value 0 and q all -inf

The spawn model is VecGame's marginal law (a uniform empty cell, a 2 with probability two_prob).  VecGame ties 2-vs-4 to the
cell within a table epoch; the search deliberately does not model that tie.
"""

from __future__ import annotations

import numpy as np

import _ntuple_ref

NEG_INF = np.float32(-np.inf)
_CHUNK = 1 << 18


def probs(two_prob: float) -> tuple[np.float32, np.float32]:
    p2 = np.float32(two_prob)
    return p2, np.float32(np.float32(1) - p2)


def _key(x: np.ndarray) -> np.ndarray:
    return np.where(np.isnan(x), NEG_INF, x).astype(np.float32)


def _value(boards: np.ndarray, weights: np.ndarray, tuples) -> np.ndarray:
    return np.concatenate([_ntuple_ref.value(boards[i:i + _CHUNK], weights, tuples) for i in range(0, boards.shape[0], _CHUNK)]
                          or [np.zeros(0, np.float32)])


def _move(move, boards: np.ndarray):
    parts = [move(boards[i:i + _CHUNK]) for i in range(0, boards.shape[0], _CHUNK)]
    if not parts:
        return np.zeros((0, 4, 16), np.uint8), np.zeros((0, 4), np.float32), np.zeros((0, 4), bool)
    return (np.concatenate([p[0] for p in parts]).astype(np.uint8), np.concatenate([p[1] for p in parts]).astype(np.float32),
            np.concatenate([p[2] for p in parts]).astype(bool))


def _argmax(key: np.ndarray, ok: np.ndarray):
    """(best direction, its key, any valid) per row: strict > in ascending direction order, so ties keep the smaller one"""
    m = key.shape[0]
    best = np.zeros(m, np.int64)
    has = ok[:, 0].copy()
    bkey = np.where(has, key[:, 0], NEG_INF).astype(np.float32)
    for a in range(1, 4):
        take = ok[:, a] & (~has | (key[:, a] > bkey))
        best = np.where(take, a, best)
        bkey = np.where(take, key[:, a], bkey).astype(np.float32)
        has |= ok[:, a]
    return best, bkey, has


def max_node(boards: np.ndarray, d: int, weights, tuples, p2, p4, move) -> np.ndarray:
    """M(b, d) for (N,16) boards: (N,) float32"""
    after, reward, valid = _move(move, boards)
    x = np.zeros(valid.shape, np.float32)
    flat = after.reshape(-1, 16)[valid.ravel()]
    inner = _value(flat, weights, tuples) if d == 1 else chance(flat, d - 1, weights, tuples, p2, p4, move)
    x[valid] = (reward[valid] + inner).astype(np.float32)
    _, bkey, has = _argmax(_key(x), valid)
    return np.where(has, bkey, np.float32(0)).astype(np.float32)


def chance(after: np.ndarray, d: int, weights, tuples, p2, p4, move) -> np.ndarray:
    """E(s, d) for (N,16) afterstates, each with at least one empty cell: (N,) float32"""
    rows, cells = np.nonzero(after == 0)  # row-major: ascending cells within each row
    n = np.bincount(rows, minlength=after.shape[0])
    assert (n >= 1).all(), "an afterstate without an empty cell"
    terms = None
    for tile, p in ((1, p2), (2, p4)):
        if p == 0:
            continue
        child = after[rows].copy()
        child[np.arange(rows.size), cells] = tile
        t = (p * max_node(child, d, weights, tuples, p2, p4, move)).astype(np.float32)
        terms = t if terms is None else (terms + t).astype(np.float32)
    # sequential per-board sums from the first term: position of each term within its board
    start = np.concatenate([[0], np.cumsum(n)[:-1]])
    pos = np.arange(rows.size) - start[rows]
    s = np.zeros(after.shape[0], np.float32)
    for k in range(int(n.max()) if n.size else 0):
        sel = pos == k
        r = rows[sel]
        s[r] = terms[sel] if k == 0 else (s[r] + terms[sel]).astype(np.float32)
    return (s / n.astype(np.float32)).astype(np.float32)


def expectimax(boards: np.ndarray, weights, tuples, *, depth: int, two_prob: float, move) -> dict:
    """the op's outputs for (M,16) uint8 boards"""
    boards = np.asarray(boards, np.uint8)
    w = np.asarray(weights, np.float32)
    p2, p4 = probs(two_prob)
    m = boards.shape[0]
    after, reward, valid = _move(move, boards)
    e = np.zeros((m, 4), np.float32)
    e[valid] = chance(after.reshape(-1, 16)[valid.ravel()], depth, w, tuples, p2, p4, move)
    q = np.full((m, 4), NEG_INF, np.float32)
    q[valid] = (reward[valid] + e[valid]).astype(np.float32)
    best, _, has = _argmax(_key(q), valid)
    rows = np.arange(m)
    return {"action": np.where(has, best, 0),
            "state": np.where(has[:, None], after[rows, best], boards),
            "reward": np.where(has, reward[rows, best], np.float32(0)).astype(np.float32),
            "value": np.where(has, e[rows, best], np.float32(0)).astype(np.float32),
            "q": q}


def oracle_move(oracle, kind: str):
    """a ``move`` over the C oracle's board_move / board_reward (exponents below 16), memoised per board"""
    memo: dict = {}

    def one(b: np.ndarray):
        key = b.tobytes()
        got = memo.get(key)
        if got is None:
            after = np.zeros((4, 16), np.uint8)
            reward = np.zeros(4, np.float32)
            valid = np.zeros(4, bool)
            for a in range(4):
                nb, mg = oracle.board_move(b, a)
                after[a] = nb
                valid[a] = bool((nb != b).any())
                reward[a] = oracle.board_reward(kind, nb, b, mg) if valid[a] else 0.0
            got = memo[key] = (after, reward, valid)
        return got

    def move(boards: np.ndarray):
        res = [one(b) for b in boards]
        return (np.stack([r[0] for r in res]) if res else np.zeros((0, 4, 16), np.uint8),
                np.stack([r[1] for r in res]) if res else np.zeros((0, 4), np.float32),
                np.stack([r[2] for r in res]) if res else np.zeros((0, 4), bool))

    return move
