"""Plain NumPy definition of delayed TD(lambda) / TC(lambda) for n-tuple networks (ml2048_b200.ops.ntuple_td_lambda_update,
ntuple_tc_lambda_update), for the tests.

Game i's window is x_0 ... x_h: x_0 the afterstate being updated, chosen h learner steps ago; x_h the one chosen this step;
rho_k (k = 1..h) the reward of the move that produced x_k; e_k (k = 0..h-1) = 1 when the environment step after x_k was chosen
ended the game; V_k = V(x_k) with the weights as they are before the call.  With lf = float32(lambda) and c = 1 - lf in
float32, every operation one float32 operation:
  R_{h-1} = e_{h-1} ? 0 : rho_h + V_h
  R_k     = e_k     ? 0 : (rho_{k+1} + c * V_{k+1}) + lf * R_{k+1}      for k = h-2 ... 0
  delta   = alpha * (R_0 - V_0)                                         (0 for a masked-out game)
The update of x_0's entries is then TD(0)'s (_ntuple_ref.td_apply_*) or TC's (_tc_ref).  Ring: after [h+1][M][16],
reward [h+1][M], ended [h+1][M]; x_k is in slot (newest - (h - k)) mod (h + 1); ended[newest] is not read.
"""

from __future__ import annotations

import numpy as np

import _ntuple_ref as nref


def lam_f32(lam: float) -> tuple[np.float32, np.float32]:
    """(lf, c) as the host rounds them"""
    lf = np.float32(lam)
    return lf, np.float32(np.float32(1) - lf)


def window(ring: np.ndarray, newest: int) -> np.ndarray:
    """ring [h+1][M]... -> the same data in window order k = 0..h"""
    slots = ring.shape[0]
    return ring[[(newest - (slots - 1 - k)) % slots for k in range(slots)]]


def lambda_return(v: np.ndarray, rho: np.ndarray, ended: np.ndarray, lam: float) -> np.ndarray:
    """R_0 (M,) float32 from window-ordered V_0..V_h (h+1, M), rho (h+1, M) (rho[0] unused) and ended (h+1, M) (ended[h]
    unused)"""
    h = v.shape[0] - 1
    lf, c = lam_f32(lam)
    v, rho, e = np.asarray(v, np.float32), np.asarray(rho, np.float32), np.asarray(ended).astype(bool)
    with np.errstate(all="ignore"):
        r = np.where(e[h - 1], np.float32(0), rho[h] + v[h]).astype(np.float32)
        for k in range(h - 2, -1, -1):
            nxt = ((rho[k + 1] + c * v[k + 1]).astype(np.float32) + (lf * r).astype(np.float32)).astype(np.float32)
            r = np.where(e[k], np.float32(0), nxt).astype(np.float32)
    return r


def lambda_delta(v: np.ndarray, rho: np.ndarray, ended: np.ndarray, lam: float, alpha: float, mask=None) -> np.ndarray:
    """delta (M,) float32 from window-ordered V, rho and ended"""
    with np.errstate(all="ignore"):
        d = (np.float32(alpha) * (lambda_return(v, rho, ended, lam) - np.asarray(v[0], np.float32))).astype(np.float32)
    if mask is not None:
        d = np.where(np.asarray(mask).astype(bool), d, np.float32(0))
    return d


def ring_delta(after_ring, reward_ring, ended_ring, newest: int, weights, tuples, lam: float, alpha: float, mask=None):
    """(delta, x_0 boards) of a ring, the values looked up with nref.value"""
    after = window(np.asarray(after_ring), newest)
    v = np.stack([nref.value(after[k], weights, tuples) for k in range(after.shape[0])])
    return lambda_delta(v, window(np.asarray(reward_ring), newest), window(np.asarray(ended_ring), newest), lam, alpha, mask), after[0]


def nstep_weighted_f64(v: np.ndarray, rho: np.ndarray, ended: np.ndarray, lam: float) -> np.ndarray:
    """(1 - l) * sum_{n=1}^{h-1} l^{n-1} G(n) + l^{h-1} G(h) in float64, l = float32(lam) exactly; G(n) = rho_1 + ... +
    rho_min(n,m) + (V_n if n <= m), m the first k with e_k (h if none): the n-step returns truncated at the first end"""
    h = v.shape[0] - 1
    lf = float(np.float32(lam))
    v, rho, e = np.asarray(v, np.float64), np.asarray(rho, np.float64), np.asarray(ended).astype(bool)
    m = np.full(v.shape[1], h)
    for k in range(h - 1, -1, -1):
        m = np.where(e[k], k, m)
    out = np.zeros(v.shape[1])
    for n in range(1, h + 1):
        g = sum(np.where(j <= m, rho[j], 0.0) for j in range(1, n + 1)) + np.where(n <= m, v[n], 0.0)
        wgt = lf ** (h - 1) if n == h else (1 - lf) * lf ** (n - 1)
        out += wgt * g
    return out
