"""Plain NumPy definition of temporal coherence learning of an n-tuple network (ml2048_b200.ops.ntuple_tc_update), for the
tests.

One synchronous batch, every operation one float32 operation.  C[j] = (E_j, A_j), the running sums of the errors applied to
entry j and of their absolute values:
  1. delta_i = alpha * (target_i - V(after_i)) with the weights before the call, 0 for a masked-out game (_ntuple_ref.td_delta);
  2. for every masked-in game and each of its 8K entries j (twice if the game hits j twice): dE_j += delta_i, dA_j += |delta_i|;
  3. for every entry with dA_j != 0 (NaN counts as non-zero), with E_j, A_j as they were before the call:
     beta_j = 1 if A_j == 0 else |E_j| / A_j;  w_j += beta_j * dE_j;  E_j += dE_j;  A_j += dA_j.
     Entries with dA_j == 0 stay as they are, bit for bit.
The device adds step 2 with float atomics (order within one entry unspecified, subnormals flushed); tc_accumulate adds in
(game, tuple, image) order, which is exact where no entry is shared between games: the repeats inside one game add equal
values, and those give the same sum in any order.
"""

from __future__ import annotations

import numpy as np

import _ntuple_ref as nref

td_delta = nref.td_delta


def tc_accumulate(after: np.ndarray, delta: np.ndarray, tuples, mask=None):
    """step 2 as sequential float32 adds in (game, t, g) order: (dE, dA), each (N,) float32"""
    n = nref.num_weights(tuples)
    de, da = np.zeros(n, np.float32), np.zeros(n, np.float32)
    keep = np.ones(after.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)
    with np.errstate(invalid="ignore", over="ignore"):
        for i, row in enumerate(nref.entries(after, tuples)):
            if keep[i]:
                d = np.float32(delta[i])
                for e in row:
                    de[e] = np.float32(de[e] + d)
                    da[e] = np.float32(da[e] + np.abs(d))
    return de, da


def tc_apply_f32(de: np.ndarray, da: np.ndarray, weights: np.ndarray, coherence: np.ndarray):
    """step 3 in float32: (weights, coherence) after the batch, new arrays"""
    w = np.array(weights, np.float32)
    c = np.array(coherence, np.float32).reshape(-1, 2)
    j = np.flatnonzero(~(da == 0))  # NaN counts as non-zero
    e0, a0 = c[j, 0], c[j, 1]
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        beta = np.where(a0 == 0, np.float32(1), np.abs(e0) / a0).astype(np.float32)
        w[j] = (w[j] + (beta * de[j]).astype(np.float32)).astype(np.float32)
        c[j, 0] = (e0 + de[j]).astype(np.float32)
        c[j, 1] = (a0 + da[j]).astype(np.float32)
    return w, c


def tc_beta_f32(coherence: np.ndarray) -> np.ndarray:
    """(N,) float32 beta of every entry as step 3 computes it from the coherence before the call"""
    c = np.asarray(coherence, np.float32).reshape(-1, 2)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(c[:, 1] == 0, np.float32(1), np.abs(c[:, 0]) / c[:, 1]).astype(np.float32)


def tc_apply_f64(after: np.ndarray, delta: np.ndarray, weights: np.ndarray, coherence: np.ndarray, tuples, mask=None):
    """steps 2 and 3 with the sums in float64 and beta as float32 computes it: (weights, E, A, adds per entry, sum |delta| per
    entry), for the tolerance of the device's atomics"""
    keep = np.ones(after.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)
    e = nref.entries(after[keep], tuples).ravel()
    d = np.repeat(delta[keep].astype(np.float64), 8 * len(tuples))
    n = nref.num_weights(tuples)
    de = np.bincount(e, weights=d, minlength=n)
    sabs = np.bincount(e, weights=np.abs(d), minlength=n)
    adds = np.bincount(e, minlength=n)
    c = np.asarray(coherence, np.float32).reshape(-1, 2)
    beta = tc_beta_f32(c).astype(np.float64)
    hit = sabs != 0
    w = np.asarray(weights, np.float64).copy()
    e64, a64 = c[:, 0].astype(np.float64), c[:, 1].astype(np.float64)
    w[hit] += beta[hit] * de[hit]
    e64[hit] += de[hit]
    a64[hit] += sabs[hit]
    return w, e64, a64, adds, sabs
