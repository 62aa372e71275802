"""Plain NumPy definition of the n-tuple network ops (ml2048_b200.ops.ntuple_*), for the tests.

Symmetries: image g of a board s holds in cell 4r+c the cell SRC[g][4r+c] of s, with (r,c) (r,3-c) (3-r,c) (3-r,3-c) (c,r)
(c,3-r) (3-c,r) (3-c,3-r) for g = 0..7.  Index: sum_j min(image[cell_j], 15) << 4j.  Value: float32 adds from 0 in the order
t = 0..K-1, g = 0..7.  Greedy: q = reward + V(afterstate) over the valid directions, NaN as -inf, ties to the smallest
direction; no valid direction -> action 0, the board itself, reward 0, value 0.  TD(0): delta = alpha * (target - V) with the
weights before the call, then w[entry] += delta for every masked-in game, tuple and image.
"""

from __future__ import annotations

import numpy as np

_SRC_RC = (lambda r, c: (r, c), lambda r, c: (r, 3 - c), lambda r, c: (3 - r, c), lambda r, c: (3 - r, 3 - c),
           lambda r, c: (c, r), lambda r, c: (c, 3 - r), lambda r, c: (3 - c, r), lambda r, c: (3 - c, 3 - r))
SRC = np.array([[4 * f(cell >> 2, cell & 3)[0] + f(cell >> 2, cell & 3)[1] for cell in range(16)] for f in _SRC_RC], np.int64)

STANDARD_4X6 = ((0, 1, 2, 3, 4, 5), (4, 5, 6, 7, 8, 9), (0, 1, 2, 4, 5, 6), (4, 5, 6, 8, 9, 10))


def offsets(tuples) -> list[int]:
    out, total = [], 0
    for t in tuples:
        out.append(total)
        total += 16 ** len(t)
    return out


def num_weights(tuples) -> int:
    return sum(16 ** len(t) for t in tuples)


def image(boards: np.ndarray, g: int) -> np.ndarray:
    """(M,16) boards -> their image g"""
    return boards[:, SRC[g]]


def index(boards: np.ndarray, cells, g: int) -> np.ndarray:
    """(M,) int64 table index of tuple `cells` on image g of every board"""
    img = np.minimum(image(boards, g).astype(np.int64), 15)
    idx = np.zeros(boards.shape[0], np.int64)
    for j, c in enumerate(cells):
        idx |= img[:, c] << (4 * j)
    return idx


def entries(boards: np.ndarray, tuples) -> np.ndarray:
    """(M, 8K) int64: every weight entry a board reads, in the value's order (t outer, g inner)"""
    offs = offsets(tuples)
    return np.stack([offs[t] + index(boards, cells, g) for t, cells in enumerate(tuples) for g in range(8)], axis=1)


def value(boards: np.ndarray, weights: np.ndarray, tuples) -> np.ndarray:
    """(M,) float32, sequential float32 adds"""
    w = np.asarray(weights, np.float32)
    acc = np.zeros(boards.shape[0], np.float32)
    for col in entries(boards, tuples).T:
        acc = acc + w[col]  # float32 + float32, one add per element, in order
    return acc


def greedy(boards: np.ndarray, after: np.ndarray, reward: np.ndarray, valid: np.ndarray, weights: np.ndarray, tuples) -> dict:
    """from afterstates (M,4,16), rewards (M,4) f32 and validity (M,4): action, state, reward, value"""
    m = boards.shape[0]
    v = value(after.reshape(-1, 16), weights, tuples).reshape(m, 4)
    q = (reward.astype(np.float32) + v).astype(np.float32)
    key = np.where(np.isnan(q), np.float32(-np.inf), q)
    ok = valid.astype(bool)
    best = np.zeros(m, np.int64)
    has = ok[:, 0].copy()
    bkey = key[:, 0].copy()
    for a in range(1, 4):
        take = ok[:, a] & (~has | (key[:, a] > bkey))  # strict: ties keep the smaller direction
        best = np.where(take, a, best)
        bkey = np.where(take, key[:, a], bkey)
        has |= ok[:, a]
    rows = np.arange(m)
    return {"action": np.where(has, best, 0),
            "state": np.where(has[:, None], after[rows, best], boards),
            "reward": np.where(has, reward[rows, best], np.float32(0)).astype(np.float32),
            "value": np.where(has, v[rows, best], np.float32(0)).astype(np.float32)}


def td_delta(after: np.ndarray, target: np.ndarray, weights: np.ndarray, tuples, alpha: float, mask=None) -> np.ndarray:
    d = (np.float32(alpha) * (target.astype(np.float32) - value(after, weights, tuples))).astype(np.float32)
    if mask is not None:
        d = np.where(np.asarray(mask).astype(bool), d, np.float32(0))
    return d


def td_apply_f32(after: np.ndarray, delta: np.ndarray, weights: np.ndarray, tuples, mask=None) -> np.ndarray:
    """phase 2 as sequential float32 adds in (game, t, g) order: exact where no entry is shared between games"""
    w = np.array(weights, np.float32)
    keep = np.ones(after.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)
    for i, row in enumerate(entries(after, tuples)):
        if keep[i]:
            for e in row:
                w[e] = np.float32(w[e] + delta[i])
    return w


def td_apply_f64(after: np.ndarray, delta: np.ndarray, weights: np.ndarray, tuples, mask=None):
    """phase 2 in float64: (weights, number of adds per entry, sum of |delta| per entry)"""
    keep = np.ones(after.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)
    e = entries(after[keep], tuples)
    d = np.repeat(delta[keep].astype(np.float64), e.shape[1])
    w = np.asarray(weights, np.float64).copy()
    np.add.at(w, e.ravel(), d)
    n = np.bincount(e.ravel(), minlength=w.size)
    s = np.bincount(e.ravel(), weights=np.abs(d), minlength=w.size)
    return w, n, s
