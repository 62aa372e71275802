"""Plain NumPy definition of weight promotion in multi-stage n-tuple networks (the ``promoted=`` argument of
ml2048_b200.ops.ntuple_*), for the tests.  Built from the staged references of _stage_ref.

promoted: N uint8 marks (N = sum_t 16^len_t, the single-stage entry count, for any S), indexed like a single-stage table.
Bit s - 1 of promoted[e] is set once stage s's entry e has been written (s = 1..S-1); stage 0 has no mark, and bits
S-1..7 are neither read nor written.

Effective weight: W(0, e) = w[e]; for s >= 1, W(s, e) = w[s * N + e] if the mark of (s, e) is set, else W(s - 1, e).  The
source stage src(s, m) is the highest k <= s with k = 0 or bit k - 1 of m set.  Every read is the staged read on W.

Update (TD(0), TC, TD(lambda), TC(lambda)): 1. the staged delta on W before the call; 2. promote: every masked-in game whose
x_0 is in stage s0 >= 1 (whatever its delta) sets, for each of its 8K entries e whose mark (s0, e) is clear,
w[s0 * N + e] = W(s0 - 1, e), for TC coherence[s0 * N + e] = (0, 0), and the mark; 3. the staged apply on x_0's own-stage
entries.  Promotion changes no effective weight.
"""

from __future__ import annotations

import numpy as np

import _ntuple_ref as nref
import _stage_ref as sref


def source_stage(s: int, m: int) -> int:
    """src(s, m): the highest k <= s with k = 0 or bit k - 1 of m set"""
    for k in range(s, 0, -1):
        if (m >> (k - 1)) & 1:
            return k
    return 0


def effective(weights, promoted, tuples, stages) -> np.ndarray:
    """(S * N,) float32 effective weights W"""
    w = np.array(weights, np.float32).reshape(sref.num_stages(stages), nref.num_weights(tuples))
    p = np.asarray(promoted, np.uint8)
    for s in range(1, w.shape[0]):
        w[s] = np.where((p >> (s - 1)) & 1 != 0, w[s], w[s - 1])
    return w.reshape(-1)


def value(boards, weights, promoted, tuples, stages) -> np.ndarray:
    return sref.value(boards, effective(weights, promoted, tuples, stages), tuples, stages)


def greedy(boards, after, reward, valid, weights, promoted, tuples, stages) -> dict:
    return sref.greedy(boards, after, reward, valid, effective(weights, promoted, tuples, stages), tuples, stages)


def expectimax(boards, weights, promoted, tuples, stages, *, depth: int, two_prob: float, move) -> dict:
    return sref.expectimax(boards, effective(weights, promoted, tuples, stages), tuples, stages, depth=depth, two_prob=two_prob,
                           move=move)


def promote(after, weights, promoted, tuples, stages, mask=None, coherence=None):
    """step 2 of an update on x_0 = ``after``: (weights, marks, coherence or None) after the promotion"""
    n = nref.num_weights(tuples)
    eff = effective(weights, promoted, tuples, stages)
    w = np.array(weights, np.float32)
    marks_before = np.asarray(promoted, np.uint8)
    marks = marks_before.copy()
    coh = None if coherence is None else np.array(coherence, np.float32)
    mask = np.ones(after.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)
    st = sref.stage(after, stages)
    ent = nref.entries(after, tuples)
    for i in np.nonzero(mask & (st >= 1))[0]:
        s0 = int(st[i])
        bit = np.uint8(1 << (s0 - 1))
        e = ent[i][(marks_before[ent[i]] & bit) == 0]
        w[s0 * n + e] = eff[(s0 - 1) * n + e]
        if coh is not None:
            coh[s0 * n + e] = 0.0
        marks[e] |= bit
    return w, marks, coh


def td_update(after, target, weights, promoted, tuples, stages, alpha, mask=None):
    """(delta, weights, marks) of one TD(0) batch; the adds in the staged reference's order"""
    d = sref.td_delta(after, target, effective(weights, promoted, tuples, stages), tuples, stages, alpha, mask)
    w, marks, _ = promote(after, weights, promoted, tuples, stages, mask)
    return d, sref.td_apply_f32(after, d, w, tuples, stages, mask), marks


def tc_update(after, target, weights, coherence, promoted, tuples, stages, alpha, mask=None):
    """(delta, weights, coherence, marks) of one TC batch"""
    d = sref.td_delta(after, target, effective(weights, promoted, tuples, stages), tuples, stages, alpha, mask)
    w, marks, coh = promote(after, weights, promoted, tuples, stages, mask, coherence)
    w, coh = sref.tc_update_f32(after, d, w, coh, tuples, stages, mask)
    return d, w, coh, marks


def lambda_update(after_ring, reward_ring, ended_ring, newest, weights, promoted, tuples, stages, lam, alpha, mask=None,
                  coherence=None):
    """(delta, weights, coherence or None, marks) of one TD(lambda) (coherence None) or TC(lambda) batch"""
    d, x0 = sref.ring_delta(after_ring, reward_ring, ended_ring, newest, effective(weights, promoted, tuples, stages), tuples,
                            stages, lam, alpha, mask)
    w, marks, coh = promote(x0, weights, promoted, tuples, stages, mask, coherence)
    if coherence is None:
        return d, sref.td_apply_f32(x0, d, w, tuples, stages, mask), None, marks
    w, coh = sref.tc_update_f32(x0, d, w, coh, tuples, stages, mask)
    return d, w, coh, marks
