"""Plain NumPy definition of multi-stage n-tuple networks (the ``stages=`` argument of ml2048_b200.ops.ntuple_*), for the
tests.  Built from the single-stage references: each of them runs on the weight slice of each board's stage.

A network has S = len(stages) + 1 stages (1..8), given by strictly ascending tile exponents tau_1 < ... < tau_{S-1} in
1..15.  m(b) = max over the 16 cells of min(b[c], 15); stage(b) = #{k : tau_k <= m(b)}: an empty board is in stage 0, a
byte >= 16 counts as 15.  The weights are S * N float32 entries (N = sum_t 16^len_t), stage s's tables at s * N in the
single-stage layout.  V(b) = sum_t sum_g w[stage(b) * N + offset_t + idx_t,g(b)], float32 adds from 0 in the single-stage
order.  Greedy values each afterstate with that afterstate's stage, expectimax each leaf with that leaf's stage, TD(lambda)
each window board x_k with that board's stage.  Every update writes the entries of x_0's stage; TC's coherence and
accumulator are (S * N, 2), indexed like the weights.  Everything else is the single-stage definition word for word.
"""

from __future__ import annotations

import numpy as np

import _expectimax_ref as xref
import _lambda_ref as lref
import _ntuple_ref as nref
import _tc_ref as tref


def num_stages(stages) -> int:
    return len(stages) + 1


def num_weights(tuples, stages) -> int:
    return num_stages(stages) * nref.num_weights(tuples)


def max_exponent(boards: np.ndarray) -> np.ndarray:
    """(M,) int64 m(b): the largest cell clamped to 15"""
    return np.minimum(np.asarray(boards, np.int64), 15).max(axis=1)


def stage(boards: np.ndarray, stages) -> np.ndarray:
    """(M,) int64 stage(b) = #{k : tau_k <= m(b)}"""
    m = max_exponent(boards)
    return (np.asarray(stages, np.int64)[None, :] <= m[:, None]).sum(axis=1) if len(stages) else np.zeros_like(m)


def _slices(weights, tuples, stages):
    """the weights as (S, N): row s is stage s's single-stage network"""
    return np.asarray(weights).reshape(num_stages(stages), nref.num_weights(tuples), *np.asarray(weights).shape[1:])


def entries(boards: np.ndarray, tuples, stages) -> np.ndarray:
    """(M, 8K) int64: every entry a board reads, in the value's order"""
    return stage(boards, stages)[:, None] * nref.num_weights(tuples) + nref.entries(boards, tuples)


def value(boards: np.ndarray, weights: np.ndarray, tuples, stages) -> np.ndarray:
    """(M,) float32: nref.value of each board on its stage's slice"""
    boards = np.asarray(boards)
    w = _slices(np.asarray(weights, np.float32), tuples, stages)
    st = stage(boards, stages)
    out = np.zeros(boards.shape[0], np.float32)
    for s in range(w.shape[0]):
        sel = st == s
        if sel.any():
            out[sel] = nref.value(boards[sel], w[s], tuples)
    return out


def greedy(boards, after, reward, valid, weights, tuples, stages) -> dict:
    """nref.greedy with every afterstate valued on its own stage's slice"""
    m = boards.shape[0]
    v = value(after.reshape(-1, 16), weights, tuples, stages).reshape(m, 4)
    q = (reward.astype(np.float32) + v).astype(np.float32)
    best, _, has = xref._argmax(xref._key(q), valid.astype(bool))
    rows = np.arange(m)
    return {"action": np.where(has, best, 0),
            "state": np.where(has[:, None], after[rows, best], boards),
            "reward": np.where(has, reward[rows, best], np.float32(0)).astype(np.float32),
            "value": np.where(has, v[rows, best], np.float32(0)).astype(np.float32)}


def _per_stage(after, tuples, stages, fn):
    """fn(selected rows, s) for every stage that some board is in"""
    st = stage(after, stages)
    for s in range(num_stages(stages)):
        sel = st == s
        if sel.any():
            fn(sel, s)


def td_delta(after, target, weights, tuples, stages, alpha, mask=None) -> np.ndarray:
    w = _slices(np.asarray(weights, np.float32), tuples, stages)
    d = np.zeros(after.shape[0], np.float32)
    mask = np.ones(after.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)

    def run(sel, s):
        d[sel] = nref.td_delta(after[sel], target[sel], w[s], tuples, alpha, mask[sel])

    _per_stage(after, tuples, stages, run)
    return d


def td_apply_f32(after, delta, weights, tuples, stages, mask=None) -> np.ndarray:
    """nref.td_apply_f32 per stage: stages own disjoint entries, so the (game, t, g) order within each is the whole order"""
    w = _slices(np.array(weights, np.float32), tuples, stages).copy()
    mask = np.ones(after.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)

    def run(sel, s):
        w[s] = nref.td_apply_f32(after[sel], delta[sel], w[s], tuples, mask[sel])

    _per_stage(after, tuples, stages, run)
    return w.reshape(-1)


def td_apply_f64(after, delta, weights, tuples, stages, mask=None):
    """nref.td_apply_f64 per stage: (weights, adds per entry, sum |delta| per entry), each (S * N,)"""
    w = _slices(np.asarray(weights, np.float64), tuples, stages).copy()
    n = np.zeros(w.shape, np.int64)
    a = np.zeros(w.shape, np.float64)
    mask = np.ones(after.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)

    def run(sel, s):
        w[s], n[s], a[s] = nref.td_apply_f64(after[sel], delta[sel], w[s], tuples, mask[sel])

    _per_stage(after, tuples, stages, run)
    return w.reshape(-1), n.reshape(-1), a.reshape(-1)


def tc_accumulate(after, delta, tuples, stages, mask=None):
    """tref.tc_accumulate per stage: (dE, dA), each (S * N,) float32"""
    n = nref.num_weights(tuples)
    de, da = np.zeros((num_stages(stages), n), np.float32), np.zeros((num_stages(stages), n), np.float32)
    mask = np.ones(after.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)

    def run(sel, s):
        de[s], da[s] = tref.tc_accumulate(after[sel], delta[sel], tuples, mask[sel])

    _per_stage(after, tuples, stages, run)
    return de.reshape(-1), da.reshape(-1)


tc_apply_f32 = tref.tc_apply_f32  # entry by entry: the stage layout does not enter


def tc_update_f32(after, delta, weights, coherence, tuples, stages, mask=None):
    """steps 2 and 3 of TC on x_0's stage: (weights, coherence) after the batch"""
    de, da = tc_accumulate(after, delta, tuples, stages, mask)
    return tc_apply_f32(de, da, weights, coherence)


def tc_apply_f64(after, delta, weights, coherence, tuples, stages, mask=None):
    """tref.tc_apply_f64 per stage: (weights, E, A, adds per entry, sum |delta| per entry), each (S * N,)"""
    n = nref.num_weights(tuples)
    w = _slices(np.asarray(weights, np.float64), tuples, stages).copy()
    c = np.asarray(coherence, np.float32).reshape(num_stages(stages), n, 2)
    e64, a64 = c[..., 0].astype(np.float64), c[..., 1].astype(np.float64)
    adds, sabs = np.zeros(w.shape, np.int64), np.zeros(w.shape, np.float64)
    mask = np.ones(after.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)

    def run(sel, s):
        w[s], e64[s], a64[s], adds[s], sabs[s] = tref.tc_apply_f64(after[sel], delta[sel], w[s], c[s], tuples, mask[sel])

    _per_stage(after, tuples, stages, run)
    return w.reshape(-1), e64.reshape(-1), a64.reshape(-1), adds.reshape(-1), sabs.reshape(-1)


def ring_delta(after_ring, reward_ring, ended_ring, newest: int, weights, tuples, stages, lam: float, alpha: float, mask=None):
    """(delta, x_0 boards) of a ring: lref.lambda_delta over values that each window board takes on its own stage"""
    after = lref.window(np.asarray(after_ring), newest)
    v = np.stack([value(after[k], weights, tuples, stages) for k in range(after.shape[0])])
    return (lref.lambda_delta(v, lref.window(np.asarray(reward_ring), newest), lref.window(np.asarray(ended_ring), newest), lam,
                              alpha, mask), after[0])


# ---- expectimax: _expectimax_ref's recursion with every leaf valued on its own stage ----------------------------------------


def _max_node(boards, d, w, tuples, stages, p2, p4, move):
    after, reward, valid = xref._move(move, boards)
    x = np.zeros(valid.shape, np.float32)
    flat = after.reshape(-1, 16)[valid.ravel()]
    inner = value(flat, w, tuples, stages) if d == 1 else _chance(flat, d - 1, w, tuples, stages, p2, p4, move)
    x[valid] = (reward[valid] + inner).astype(np.float32)
    _, bkey, has = xref._argmax(xref._key(x), valid)
    return np.where(has, bkey, np.float32(0)).astype(np.float32)


def _chance(after, d, w, tuples, stages, p2, p4, move):
    rows, cells = np.nonzero(after == 0)
    n = np.bincount(rows, minlength=after.shape[0])
    assert (n >= 1).all(), "an afterstate without an empty cell"
    terms = None
    for tile, p in ((1, p2), (2, p4)):
        if p == 0:
            continue
        child = after[rows].copy()
        child[np.arange(rows.size), cells] = tile
        t = (p * _max_node(child, d, w, tuples, stages, p2, p4, move)).astype(np.float32)
        terms = t if terms is None else (terms + t).astype(np.float32)
    start = np.concatenate([[0], np.cumsum(n)[:-1]])
    pos = np.arange(rows.size) - start[rows]
    s = np.zeros(after.shape[0], np.float32)
    for k in range(int(n.max()) if n.size else 0):
        sel = pos == k
        r = rows[sel]
        s[r] = terms[sel] if k == 0 else (s[r] + terms[sel]).astype(np.float32)
    return (s / n.astype(np.float32)).astype(np.float32)


def expectimax(boards, weights, tuples, stages, *, depth: int, two_prob: float, move) -> dict:
    """xref.expectimax's outputs with every leaf valued on its own stage"""
    boards = np.asarray(boards, np.uint8)
    w = np.asarray(weights, np.float32)
    p2, p4 = xref.probs(two_prob)
    m = boards.shape[0]
    after, reward, valid = xref._move(move, boards)
    e = np.zeros((m, 4), np.float32)
    e[valid] = _chance(after.reshape(-1, 16)[valid.ravel()], depth, w, tuples, stages, p2, p4, move)
    q = np.full((m, 4), xref.NEG_INF, np.float32)
    q[valid] = (reward[valid] + e[valid]).astype(np.float32)
    best, _, has = xref._argmax(xref._key(q), valid)
    rows = np.arange(m)
    return {"action": np.where(has, best, 0),
            "state": np.where(has[:, None], after[rows, best], boards),
            "reward": np.where(has, reward[rows, best], np.float32(0)).astype(np.float32),
            "value": np.where(has, e[rows, best], np.float32(0)).astype(np.float32),
            "q": q}
