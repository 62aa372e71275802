"""Plain high-precision references of the floating-point rollout ops, shared by the host-shim tests (CPU) and
tests/test_rollout_numerics.py (GPU):

    policy_words            the policy's uniform word of a global slot (board_ops.cuh: slot_word, stream tag 0), NumPy
    ref_masked_categorical  the masked categorical sample in float64: inverse-CDF action, log_softmax, distance to a boundary
    check_sampler           the acceptance rules of a sampler's (action, log-prob) output against that reference
    sampler_logits          the logit classes the rules are checked on
    ref_gae                 compute_gae's recurrence (gae.py:50, :65-68) in torch float32, the op order of the reference
"""

from __future__ import annotations

from types import SimpleNamespace

import numpy as np

M32 = 0xFFFFFFFF
FMIN32 = float(np.finfo(np.float32).min)  # what the reference writes over invalid actions (policy/actor_critic.py:56-76)
BOUNDARY_TOL = 4.0 / 2**24                # |u - CDF boundary| below which either neighbouring action is accepted
LOGIT_CLASSES = ("randn3", "dominant", "pm1e4", "pm1e30", "ties", "boundary")  # see sampler_logits


def philox2x32_10(c0, c1, key):
    """Philox2x32-10 (Random123), vectorised over the counter words; `key` is a Python int."""
    c0 = np.asarray(c0, np.uint64) & M32
    c1 = np.asarray(c1, np.uint64) & M32
    k = np.uint64(key & M32)
    for _ in range(10):
        p = c0 * np.uint64(0xD256D193)
        c0, c1 = (p >> np.uint64(32)) ^ k ^ c1, p & np.uint64(M32)
        k = (k + np.uint64(0x9E3779B9)) & np.uint64(M32)
    return c0.astype(np.uint32), c1.astype(np.uint32)


def policy_words(slot, counter: int, seed: int) -> np.ndarray:
    """slot_word(slot, counter, seed, tag=0) for an array of global slots: one half of the Philox2x32-10 block of the slot
    pair (slot >> 1, block_counter_word(slot >> 1, counter)) under key stream_key(seed, 0); even slot -> .x, odd -> .y."""
    slot = np.asarray(slot, np.uint64)
    key = (seed & M32) ^ (((seed >> 32) * 0x9E3779B9) & M32)
    pair = slot >> np.uint64(1)
    ctr_word = np.uint64((counter & M32) ^ (((counter >> 32) * 0x85EBCA6B) & M32))
    c1 = ctr_word ^ (((pair >> np.uint64(32)) * np.uint64(0xC2B2AE35)) & np.uint64(M32))
    x, y = philox2x32_10(pair & np.uint64(M32), c1, key)
    return np.where((slot & np.uint64(1)) == 1, y, x)


def uniform_of(words) -> np.ndarray:
    """The sampler's uniform in [0, 1): the top 24 bits of the word."""
    return (np.asarray(words, np.uint32) >> 8).astype(np.float64) / 2**24


def ref_masked_categorical(logits, valid, words) -> SimpleNamespace:
    """float64 reference of the masked categorical sample of (n, 4) float32 logits, (n, 4) masks (nonzero = valid) and (n,)
    uniform words.  Invalid actions take finfo(float32).min as the reference does, so a row whose valid logits are all -inf
    (or that has none valid) draws from the masked actions.  Returns action (inverse CDF: #{k : u >= C_k}), log_prob
    (log_softmax, every action), p, cdf, u and boundary_dist (distance of u to the nearest CDF boundary with probability
    mass on both sides, inf when there is none)."""
    l = np.where(np.asarray(valid) != 0, np.asarray(logits, np.float32).astype(np.float64), FMIN32)
    with np.errstate(invalid="ignore", over="ignore"):
        mx = l.max(axis=1, keepdims=True)
        e = np.exp(l - mx)
        total = e.sum(axis=1, keepdims=True)
        log_prob = l - (mx + np.log(total))
        p = e / total
    cdf = np.cumsum(p, axis=1)
    after = np.cumsum(p[:, ::-1], axis=1)[:, ::-1] - p  # mass strictly after action k
    u = uniform_of(words)
    action = np.minimum((u[:, None] >= cdf).sum(axis=1), 3)
    interior = (cdf > 0) & (after > 0)
    boundary_dist = np.where(interior, np.abs(u[:, None] - cdf), np.inf).min(axis=1)
    return SimpleNamespace(action=action, log_prob=log_prob, p=p, cdf=cdf, u=u, boundary_dist=boundary_dist)


def check_sampler(logits, valid, words, actions, log_probs, *, adversarial: bool = False, what: str = "") -> dict:
    """Assert a sampler's outputs against ref_masked_categorical on every row with at least one valid finite logit above
    finfo.min and no valid NaN / +inf logit:

      action    == the reference's, or, when u lies within BOUNDARY_TOL of a CDF boundary, the action on either side of
                   it; always a valid action with p > 0
      log-prob  |lp - ref_lp[a]| <= 2^-22 (|l_a| + |max valid logit|) + 2^-21: the rounding of l_a - logsumexp in fp32
                scales with the logits

    Rows near a boundary must be rare unless the class is built to hit boundaries (`adversarial`).  Returns counts and the
    largest log-prob error as a fraction of its tolerance."""
    logits = np.asarray(logits, np.float32)
    v = np.asarray(valid) != 0
    a = np.asarray(actions).astype(np.int64)
    lp = np.asarray(log_probs, np.float32).astype(np.float64)
    ref = ref_masked_categorical(logits, v, words)
    finite = v & np.isfinite(logits) & (logits > FMIN32)
    poisoned = v & (np.isnan(logits) | (logits == np.inf))
    rows = np.flatnonzero(finite.any(axis=1) & ~poisoned.any(axis=1))
    ar = a[rows]
    assert ((ar >= 0) & (ar <= 3)).all(), (what, "action out of range")
    ok_valid = v[rows, ar] & (ref.p[rows, ar] > 0)
    bad = np.flatnonzero(~ok_valid)
    assert bad.size == 0, (what, "invalid or impossible action", rows[bad[0]], logits[rows[bad[0]]], v[rows[bad[0]]], ar[bad[0]])
    u = ref.u[rows]
    near = ref.boundary_dist[rows] <= BOUNDARY_TOL
    lo = np.where(ar > 0, ref.cdf[rows, np.maximum(ar - 1, 0)], 0.0)
    hi = ref.cdf[rows, ar]
    ok = (ar == ref.action[rows]) | (near & (lo - BOUNDARY_TOL <= u) & (u < hi + BOUNDARY_TOL))
    bad = np.flatnonzero(~ok)
    if bad.size:
        r = rows[bad[0]]
        raise AssertionError(f"{what}: {bad.size} wrong actions; row {r}: logits {logits[r]} valid {v[r]} u {ref.u[r]!r} "
                             f"cdf {ref.cdf[r]} got {a[r]} want {ref.action[r]} boundary_dist {ref.boundary_dist[r]:.3g}")
    lmax = np.where(finite, logits, -np.inf).max(axis=1)[rows].astype(np.float64)
    la = logits[rows, ar].astype(np.float64)
    tol = 2.0**-22 * (np.abs(la) + np.abs(lmax)) + 2.0**-21
    err = np.abs(lp[rows] - ref.log_prob[rows, ar])
    bad = np.flatnonzero(~(err <= tol))
    if bad.size:
        r = rows[bad[0]]
        raise AssertionError(f"{what}: {bad.size} log-probs off; row {r}: logits {logits[r]} valid {v[r]} action {a[r]} "
                             f"lp {lp[r]!r} want {ref.log_prob[r, a[r]]!r} tol {tol[bad[0]]:.3g}")
    n_near = int(near.sum())
    if not adversarial:
        assert n_near <= 4 + 1e-4 * rows.size, (what, "boundary rows are not rare", n_near, rows.size)
    return {"rows": int(rows.size), "boundary_rows": n_near, "max_lp_err_over_tol": float((err / tol).max()) if rows.size else 0.0}


def sampler_logits(name: str, rng: np.random.Generator, words: np.ndarray) -> np.ndarray:
    """(n, 4) float32 logits of class `name` (LOGIT_CLASSES) for the rows that will be sampled with `words` (the boundary
    class needs them).  Every class is checked with check_sampler; "boundary" is adversarial, and its masks must keep
    actions 0 and 1 valid (boundary_valid)."""
    n = words.shape[0]
    if name == "randn3":
        x = rng.standard_normal((n, 4)) * 3
    elif name == "dominant":  # the others 80-120 below: their expf underflows to subnormal / zero in fp32
        x = -rng.uniform(80.0, 120.0, (n, 4))
        x[np.arange(n), rng.integers(0, 4, n)] = 0.0
        x += rng.standard_normal((n, 1)) * 10
    elif name == "pm1e4":
        x = rng.choice([-1e4, 1e4], (n, 1)) + rng.standard_normal((n, 4))
    elif name == "pm1e30":
        x = np.where(rng.random((n, 1)) < 0.5, rng.standard_normal((n, 4)) * 1e30,
                     rng.choice([-1e30, 1e30], (n, 1)) * (1 + rng.integers(0, 3, (n, 4)) * 1e-7))
    elif name == "ties":
        x = np.round(rng.standard_normal((n, 4)))  # partial ties, and rows of four equal logits
        whole = rng.random(n) < 0.5
        x[whole] = rng.choice([0.0, -3.5, 17.25, 1e30, -1e4], (int(whole.sum()), 1))
    elif name == "boundary":  # p0 == u: u sits on the first CDF boundary up to the rounding of the logits to fp32
        u = uniform_of(words)
        with np.errstate(divide="ignore"):
            x = np.stack([np.log(u), np.log1p(-u), np.full(n, -np.inf), np.full(n, -np.inf)], axis=1)
    else:
        raise ValueError(name)
    return np.ascontiguousarray(x, dtype=np.float32)


def boundary_valid(valid: np.ndarray) -> np.ndarray:
    """The masks of the boundary class: actions 0 and 1 valid (their bytes kept when nonzero), 2 and 3 as given."""
    v = valid.copy()
    v[:, :2] = np.where(v[:, :2] != 0, v[:, :2], 1)
    return v


def random_masks(rng: np.random.Generator, n: int, wide: bool = True) -> np.ndarray:
    """(n, 4) uint8 masks over all 16 patterns; with `wide`, the valid bytes of half the rows hold 2..255 instead of 1."""
    bits = rng.integers(0, 16, n)
    v = ((bits[:, None] >> np.arange(4)) & 1).astype(np.uint8)
    if wide:
        big = (rng.random((n, 1)) < 0.5) & (v != 0)
        v = np.where(big, rng.integers(2, 256, (n, 4)), v).astype(np.uint8)
    return v


def _kth_valid(v: np.ndarray, k: np.ndarray) -> np.ndarray:
    rank = np.cumsum(v, axis=1) - 1
    return np.argmax(v & (rank == k[:, None]), axis=1)


def check_sampler_exact(sample, words: np.ndarray, rng: np.random.Generator) -> None:
    """The cases a sampler must get exactly right, for `sample(logits, valid) -> (actions, log_probs)` drawing row i with
    words[i] (NumPy in and out; the rows are len(words)):

      one valid action             that action, log-prob 0
      no valid action              action word >> 30 (the reference draws uniformly over the masked ones), log-prob 0
      k valid actions, equal logits   the floor(k u)-th valid action
      masked logit NaN / +-inf     bit-identical outputs to the same row with that logit 0
      valid -inf next to a finite  that action is never drawn (and the other rules hold)
      valid NaN / +inf             log-prob NaN, never a silently finite value; action in 0..3"""
    n = words.shape[0]
    f = np.float32
    w = words.astype(np.int64)
    rows = np.arange(n)
    scale = rng.choice([1.0, 1e4, 1e30], (n, 1))
    junk = rng.choice(np.array([0.0, np.nan, np.inf, -np.inf, 5.0], f), (n, 4))  # what masked actions hold

    def run(logits, valid):
        a, lp = sample(np.ascontiguousarray(logits, f), np.ascontiguousarray(valid, np.uint8))
        return np.asarray(a).astype(np.int64), np.asarray(lp, f)

    # one valid action
    only = rng.integers(0, 4, n)
    v = np.zeros((n, 4), np.uint8)
    v[rows, only] = rng.integers(1, 256, n)
    a, lp = run(np.where(v != 0, rng.standard_normal((n, 4)) * scale, junk), v)
    np.testing.assert_array_equal(a, only, err_msg="one valid action")
    assert (lp == 0.0).all(), ("one valid action: log-prob", lp[lp != 0.0][:4])

    # no valid action
    v = np.zeros((n, 4), np.uint8)
    a, lp = run(np.where(rng.random((n, 4)) < 0.5, junk, rng.standard_normal((n, 4)) * scale), v)
    np.testing.assert_array_equal(a, w >> 30, err_msg="no valid action")
    assert (lp == 0.0).all(), ("no valid action: log-prob", lp[lp != 0.0][:4])

    # equal logits over the k valid actions; a word within 3 * 2^-24 of 1/3 or 2/3 gets three valid actions: there the
    # 24th bit of the uniform decides the action (a 23-bit uniform draws floor(3 u) - 1 at u = 0xAAAAAB / 2^24)
    v = random_masks(rng, n)
    v[(v != 0).sum(axis=1) == 0, rng.integers(0, 4)] = 1
    r3 = (3 * (w >> 8)) % (1 << 24)
    third = (r3 <= 3) | (r3 >= (1 << 24) - 3)
    v[third] = np.array([[1, 1, 1, 0], [1, 1, 0, 1], [1, 0, 1, 1], [0, 1, 1, 1]], np.uint8)[rng.integers(0, 4, int(third.sum()))]
    k = (v != 0).sum(axis=1)
    level = rng.choice([0.0, -7.5, 3.25, 1e4, -1e30, 1e30], (n, 1))
    a, lp = run(np.where(v != 0, level, junk), v)
    np.testing.assert_array_equal(a, _kth_valid(v != 0, (k * (w >> 8)) >> 24), err_msg="equal logits")

    # masked logits: NaN / +inf / -inf behave exactly like 0
    v = random_masks(rng, n)
    v[(v != 0).all(axis=1), rng.integers(0, 4)] = 0
    base = np.where(v != 0, rng.standard_normal((n, 4)) * scale, 0.0)
    a0, lp0 = run(base, v)
    for val in (np.nan, np.inf, -np.inf):
        a, lp = run(np.where(v != 0, base, val), v)
        np.testing.assert_array_equal(a, a0, err_msg=f"masked {val}")
        np.testing.assert_array_equal(lp.view(np.uint32), lp0.view(np.uint32), err_msg=f"masked {val}")

    # a valid -inf logit next to finite ones is never drawn
    v = random_masks(rng, n)
    few = (v != 0).sum(axis=1) < 2
    v[few, :2] = 1
    dead = _kth_valid(v != 0, rng.integers(0, 2, n))
    logits = (rng.standard_normal((n, 4)) * scale).astype(f)
    logits[rows, dead] = -np.inf
    a, lp = run(logits, v)
    assert (a != dead).all(), "a valid -inf logit was drawn"
    check_sampler(logits, v, words, a, lp, what="valid -inf")

    # a valid NaN or +inf logit poisons the log-prob
    v = random_masks(rng, n)
    v[(v != 0).sum(axis=1) == 0, rng.integers(0, 4)] = 1
    bad = _kth_valid(v != 0, rng.integers(0, 4, n) % (v != 0).sum(axis=1))
    logits = (rng.standard_normal((n, 4)) * 3).astype(f)
    logits[rows, bad] = rng.choice(np.array([np.nan, np.inf], f), n)
    a, lp = run(logits, v)
    assert ((a >= 0) & (a <= 3)).all()
    assert np.isnan(lp).all(), ("valid NaN / +inf: finite log-prob", lp[~np.isnan(lp)][:4])


def ref_gae(v0, v1, reward, terminated, gamma: float, lambda_: float):
    """compute_gae (gae.py:50, :65-68) in torch float32, op for op: delta = gamma * v1 * mask + reward - v0, then the
    reverse scan tmp = delta[t] + (tmp * (gamma * lambda_)) * mask[t].  `terminated` is bool or uint8 (nonzero = ended)."""
    import torch

    mask = terminated == 0
    delta = gamma * v1 * mask + reward - v0
    u, s, n = v0.shape
    tmp = torch.zeros(u, n, dtype=v0.dtype, device=v0.device)
    out = torch.empty_like(v0)
    for idx in reversed(range(s)):
        tmp = tmp * (gamma * lambda_)
        tmp = delta[:, idx, :] + tmp * mask[:, idx, :]
        out[:, idx, :] = tmp
    return out
