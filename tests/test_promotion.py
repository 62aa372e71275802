"""
Weight promotion of multi-stage n-tuple networks on the GPU (the ``promoted=`` argument of ``ops.ntuple_*``,
``NTupleNetwork(..., promotion=True)``) against the NumPy definition in tests/_promotion_ref.py.

- Reads at S = 2, 3 and 8 with random marks: value, greedy (uint8 and int64 actions) and expectimax depth 1 and 2 bit for
  bit against the reference and against the staged op on ``ntuple_promoted_weights``; the same again with the storage of
  every unmarked entry poisoned with NaN.
- Updates (TD(0), TC, TD(lambda), TC(lambda)) on integer data: weights, coherence, marks and delta bit for bit, canaries
  around every buffer, stage 0 and the stages no x_0 is in untouched; crafted boards that hit one entry in two or three
  stages within one call; a second call promotes nothing new.
- The promote kernel's race at scale: M = 2^20 + 3 games over 2048 race boards in stages 1..7 of S = 8, every mark clear
  and NaN behind it; alpha = 0 (promotion only) bit for bit for all four rules, a second call promotes nothing, then one
  alpha = 1/16 call whose every partial sum is exact, bit for bit.
- All marks set is the staged op bit for bit and leaves the marks; S = 1 with marks is the single-stage op bit for bit.
- CUDA-graph replay of greedy + each update equals eager; the learner, state_dict's three load rules and both policies.
"""

from __future__ import annotations

import numpy as np
import pytest
import torch

import _ntuple_ref as nref
import _promotion_ref as pref
import _stage_ref as sref
from _ntuple_gpu import _gpu, ops  # noqa: F401 (ops is a fixture)
from test_stages import (CASES, KINDS, SMALL, _afterstate_move, _crossing_boards, _edge_boards, _guarded, _same_bits,
                         _stage_weights, played)  # noqa: F401 (played is a fixture)


def _marks(rng, n: int, stages) -> np.ndarray:
    """random marks with bits S-1..7 random too (they must be ignored)"""
    return rng.integers(0, 256, n, dtype=np.uint8)


def _poisoned(w: np.ndarray, marks: np.ndarray, tuples, stages) -> np.ndarray:
    n = nref.num_weights(tuples)
    p = w.copy().reshape(len(stages) + 1, n)
    for s in range(1, len(stages) + 1):
        p[s][(marks >> (s - 1)) & 1 == 0] = np.nan
    return p.reshape(-1)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_reads_bit_exact(ops, played, case):
    dev = _gpu()
    stages, tuples = CASES[case]
    rng = np.random.default_rng(100 + list(CASES).index(case))
    n = nref.num_weights(tuples)
    w = _stage_weights(rng, tuples, stages)
    marks = _marks(rng, n, stages)
    pm = torch.from_numpy(marks).to(dev)
    boards = np.concatenate([played, _edge_boards(rng, stages), _crossing_boards(stages)])
    b = torch.from_numpy(boards).to(dev)
    for wi in (w, _poisoned(w, marks, tuples, stages)):
        w_dev = torch.from_numpy(wi).to(dev)
        eff = ops.ntuple_promoted_weights(w_dev, pm, tuples, stages)
        _same_bits(eff.cpu().numpy(), pref.effective(w, marks, tuples, stages), "effective weights")
        got = ops.ntuple_value(b, w_dev, tuples, stages=stages, promoted=pm).cpu().numpy()
        _same_bits(got, pref.value(boards, w, marks, tuples, stages), "value")
        _same_bits(got, ops.ntuple_value(b, eff, tuples, stages=stages).cpu().numpy(), "value vs staged")
        for kind in KINDS[:2]:
            after, reward, valid = _afterstate_move(ops, kind)(boards)
            want = pref.greedy(boards, after, reward, valid, w, marks, tuples, stages)
            for dtype in (torch.uint8, torch.int64):
                g = ops.ntuple_greedy(b, w_dev, tuples, reward_fn=kind, action_dtype=dtype, stages=stages, promoted=pm)
                s = ops.ntuple_greedy(b, eff, tuples, reward_fn=kind, action_dtype=dtype, stages=stages)
                np.testing.assert_array_equal(g["action"].cpu().numpy().astype(np.int64), want["action"])
                np.testing.assert_array_equal(g["state"].cpu().numpy(), want["state"])
                for k in ("reward", "value"):
                    _same_bits(g[k].cpu().numpy(), want[k], k)
                for k in g:
                    assert torch.equal(g[k].view(torch.uint8), s[k].view(torch.uint8)), k
        for depth in (1, 2):
            pool = np.concatenate([_crossing_boards(stages), played[rng.permutation(played.shape[0])[:24 if depth == 2 else 300]]])
            want = pref.expectimax(pool, w, marks, tuples, stages, depth=depth, two_prob=0.9, move=_afterstate_move(ops, "normal"))
            bp = torch.from_numpy(pool).to(dev)
            got = ops.ntuple_expectimax(bp, w_dev, tuples, depth=depth, two_prob=0.9, stages=stages, promoted=pm)
            st = ops.ntuple_expectimax(bp, eff, tuples, depth=depth, two_prob=0.9, stages=stages)
            np.testing.assert_array_equal(got["action"].cpu().numpy(), want["action"])
            for k in ("reward", "value", "q"):
                _same_bits(got[k].cpu().numpy(), want[k], f"expectimax{depth} {k}")
            for k in got:
                assert torch.equal(got[k].view(torch.uint8), st[k].view(torch.uint8)), k
    assert torch.equal(pm.cpu(), torch.from_numpy(marks)), "a read wrote the marks"


def _race_boards(stages, tuples, bases: int = 24, seed: int = 7) -> np.ndarray:
    """boards with identical tuple cells but their largest tile outside every tuple, one per stage: the same entry e of
    several stages in one call"""
    cells = sorted({c for t in tuples for c in t})
    free = [c for c in range(16) if c not in cells]
    assert free, "every cell is in a tuple"
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(bases):
        base = np.zeros(16, np.uint8)
        base[cells] = rng.integers(0, 2, len(cells))
        for top in [1] + list(stages):
            b = base.copy()
            b[free[0]] = top
            out.append(b)
    return np.stack(out)


RACE_TUPLES = ((0, 1, 2, 3), (4, 5, 6, 7))  # cells 8..15 free for the largest tile


def _run_update(ops, rule, dev, x_or_ring, target, w_dev, c_dev, acc, tuples, stages, pm, mk, d_dev, alpha):
    if rule in ("td0", "tc"):
        a = torch.from_numpy(x_or_ring).to(dev)
        t = torch.from_numpy(target).to(dev)
        if rule == "td0":
            ops.ntuple_td_update(a, t, w_dev, tuples, alpha=alpha, mask=mk, delta_out=d_dev, stages=stages, promoted=pm)
        else:
            ops.ntuple_tc_update(a, t, w_dev, c_dev, acc, tuples, alpha=alpha, mask=mk, delta_out=d_dev, stages=stages, promoted=pm)
        return
    ring, rew, ended = x_or_ring
    args = (torch.from_numpy(ring).to(dev), torch.from_numpy(rew).to(dev), torch.from_numpy(ended).to(dev), 1)
    if rule == "lambda_td":
        ops.ntuple_td_lambda_update(*args, w_dev, tuples, alpha=alpha, lam=0.5, mask=mk, delta_out=d_dev, stages=stages, promoted=pm)
    else:
        ops.ntuple_tc_lambda_update(*args, w_dev, c_dev, acc, tuples, alpha=alpha, lam=0.5, mask=mk, delta_out=d_dev, stages=stages,
                                    promoted=pm)


def _want_update(rule, x_or_ring, target, w, coh, marks, tuples, stages, mask, alpha):
    if rule == "td0":
        d, w2, m2 = pref.td_update(x_or_ring, target, w, marks, tuples, stages, alpha, mask)
        return d, w2, None, m2
    if rule == "tc":
        return pref.tc_update(x_or_ring, target, w, coh, marks, tuples, stages, alpha, mask)
    ring, rew, ended = x_or_ring
    return pref.lambda_update(ring, rew, ended, 1, w, marks, tuples, stages, 0.5, alpha, mask,
                              coh if rule == "lambda_tc" else None)


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc", "lambda_td", "lambda_tc"])
@pytest.mark.parametrize("case", list(CASES) + ["race"])
def test_updates_exact(ops, played, case, rule):
    """integer weights and targets, alpha = 1/16, lambda = 1/2: every sum exact, so the atomics' order cannot change a bit"""
    dev = _gpu()
    stages, tuples = ((3, 5), RACE_TUPLES) if case == "race" else CASES[case]
    rng = np.random.default_rng(200 + (list(CASES) + ["race"]).index(case))
    n = nref.num_weights(tuples)
    S = len(stages) + 1
    pool = _race_boards(stages, tuples) if case == "race" else np.concatenate([played, _edge_boards(rng, stages)])
    alpha = 0.0625
    lam_rule = rule.startswith("lambda")
    m = 1500 if lam_rule else pool.shape[0]
    if lam_rule:
        ring = pool[rng.integers(0, pool.shape[0], size=(3 + 1, m))]
        if case == "race":
            ring[2] = pool[np.arange(m) % pool.shape[0]]
        data = (ring, rng.choice(np.array([0, 4, 8, 256], np.float32), size=(4, m)), (rng.random((4, m)) < 0.1).astype(np.uint8))
        x0 = ring[2]  # newest = 1, h = 3: x_0 in slot 2
    else:
        data = x0 = pool
    w = _stage_weights(rng, tuples, stages, integer=True)
    target = rng.integers(-64, 65, size=m).astype(np.float32)
    mask = (rng.random(m) < 0.8).astype(np.uint8)
    coh = rng.integers(-20, 21, size=(w.size, 2)).astype(np.float32)
    coh[:, 1] = np.abs(coh[:, 1]) + np.abs(coh[:, 0])
    marks = _marks(rng, n, stages)
    if case == "race":
        marks[:] = 0
        assert len(set(sref.stage(x0[mask.astype(bool)], stages).tolist()) - {0}) >= 2
    tc = rule in ("tc", "lambda_tc")
    w_dev, w_ok = _guarded((w.size,), torch.float32, dev, torch.from_numpy(w))
    pm, pm_ok = _guarded((n,), torch.uint8, dev, torch.from_numpy(marks))
    d_dev, d_ok = _guarded((m,), torch.float32, dev)
    c_dev, c_ok = _guarded((w.size, 2), torch.float32, dev, torch.from_numpy(coh))
    acc, acc_ok = _guarded((w.size, 2), torch.float32, dev, torch.zeros((w.size, 2)))
    mk = torch.from_numpy(mask).to(dev)
    for call in range(2):
        w_dev.copy_(torch.from_numpy(w))  # integer weights again: a TC step leaves fractions, and then the order of adds counts
        c_dev.copy_(torch.from_numpy(coh))
        w_before, m_before = w_dev.cpu().numpy(), pm.cpu().numpy()
        c_before = c_dev.cpu().numpy()
        want_d, want_w, want_c, want_m = _want_update(rule, data, target, w_before, c_before, m_before, tuples, stages, mask, alpha)
        _run_update(ops, rule, dev, data, target, w_dev, c_dev, acc, tuples, stages, pm, mk, d_dev, alpha)
        _same_bits(d_dev.cpu().numpy(), want_d, "delta")
        got_w, got_m = w_dev.cpu().numpy(), pm.cpu().numpy()
        _same_bits(got_w, want_w, "weights")
        np.testing.assert_array_equal(got_m, want_m, "marks")
        if tc:
            _same_bits(c_dev.cpu().numpy(), want_c, "coherence")
        else:
            assert torch.equal(c_dev.cpu(), torch.from_numpy(c_before))
        assert not bool(acc.view(torch.int32).any())
        # bits S-1..7 as they were; stage 0 written only by the apply; untouched stages bit for bit
        high = np.uint8((0xFF << (S - 1)) & 0xFF)
        np.testing.assert_array_equal(got_m & high, m_before & high)
        hit = set(sref.stage(x0[mask.astype(bool)], stages).tolist())
        for s in range(S):
            if s not in hit:
                np.testing.assert_array_equal(got_w[s * n:(s + 1) * n].view(np.uint32), w_before[s * n:(s + 1) * n].view(np.uint32))
        if call == 0:
            assert (got_m != m_before).any(), "nothing was promoted"
        else:
            np.testing.assert_array_equal(got_m, m_before, "a second call promoted something new")
    for ok in (w_ok, pm_ok, d_ok, c_ok, acc_ok):
        ok()


def _race_call(ops, rule, dev, x0, k, w_dev, c_dev, acc, tuples, stages, pm, mk, d_dev, alpha):
    """one update whose every x_0 is x0 and whose delta is alpha * k: TD(0) / TC toward V(x0) + k; the lambda rules with
    h = 1, x_1 = x_0 and reward k, whose return is then k + V(x0) as well"""
    b = torch.from_numpy(x0).to(dev)
    kk = torch.from_numpy(k).to(dev)
    kw = dict(alpha=alpha, mask=mk, delta_out=d_dev, stages=stages, promoted=pm)
    if rule in ("td0", "tc"):
        target = ops.ntuple_value(b, w_dev, tuples, stages=stages, promoted=pm) + kk
        if rule == "td0":
            ops.ntuple_td_update(b, target, w_dev, tuples, **kw)
        else:
            ops.ntuple_tc_update(b, target, w_dev, c_dev, acc, tuples, **kw)
        return
    ring = (torch.stack([b, b]), torch.stack([kk, kk]), torch.zeros((2, b.shape[0]), dtype=torch.uint8, device=dev), 1)
    if rule == "lambda_td":
        ops.ntuple_td_lambda_update(*ring, w_dev, tuples, lam=0.5, **kw)
    else:
        ops.ntuple_tc_lambda_update(*ring, w_dev, c_dev, acc, tuples, lam=0.5, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc", "lambda_td", "lambda_tc"])
def test_promotion_race_at_scale(ops, rule):
    """M = 2^20 + 3 games over 2048 race boards (256 bases, one board per stage 1..7 of S = 8), so that every entry is met by
    many games in several stages within one launch, from clear marks and NaN behind every one of them.

    alpha = 0: the call only promotes, and what it promotes does not depend on the order in which the games meet an entry,
    so weights, marks and coherence must equal the reference bit for bit; no touched effective weight is NaN; a second call
    promotes nothing.  Then one alpha = 1/16 call, again from clear marks, with delta = k / 16 (k in {-1, 0, 1}): every
    partial sum of an entry is a multiple of 1/16 below 2^24 / 16 (asserted), so it is exact in any order, and weights,
    coherence and marks are bit for bit too.  4.7 s per rule on one B200 (power limit not recorded), most of it the host
    reference."""
    dev = _gpu()
    stages, tuples = tuple(range(1, 8)), RACE_TUPLES
    n = nref.num_weights(tuples)
    rng = np.random.default_rng(600 + ["td0", "tc", "lambda_td", "lambda_tc"].index(rule))
    pool = _race_boards(stages, tuples, bases=256, seed=11)
    m = (1 << 20) + 3
    x0 = pool[rng.integers(0, pool.shape[0], m)]
    mask = (rng.random(m) < 0.9).astype(np.uint8)
    keep = mask.astype(bool)
    assert set(sref.stage(x0[keep], stages).tolist()) == set(range(1, 8))
    distinct = np.unique(x0[keep], axis=0)  # promotion is idempotent: duplicates of a board promote nothing more
    w = _poisoned(_stage_weights(rng, tuples, stages, integer=True), np.zeros(n, np.uint8), tuples, stages)
    coh = rng.integers(-20, 21, size=(w.size, 2)).astype(np.float32)
    coh[:, 1] = np.abs(coh[:, 1]) + np.abs(coh[:, 0])
    tc = rule in ("tc", "lambda_tc")
    w_dev = torch.from_numpy(w).to(dev)
    c_dev = torch.from_numpy(coh).to(dev)
    acc = torch.zeros((w.size, 2), device=dev)
    pm = torch.zeros(n, dtype=torch.uint8, device=dev)
    mk = torch.from_numpy(mask).to(dev)
    d_dev = torch.empty(m, device=dev)
    k = rng.integers(-1, 2, size=m).astype(np.float32)
    want_w, want_m, want_c = pref.promote(distinct, w, np.zeros(n, np.uint8), tuples, stages, None, coh if tc else None)
    ent = sref.entries(distinct, tuples, stages)
    for call in range(2):
        _race_call(ops, rule, dev, x0, k, w_dev, c_dev, acc, tuples, stages, pm, mk, d_dev, 0.0)
        _same_bits(w_dev.cpu().numpy(), want_w, f"weights, call {call}")
        np.testing.assert_array_equal(pm.cpu().numpy(), want_m, f"marks, call {call}")
        _same_bits(c_dev.cpu().numpy(), want_c if tc else coh, f"coherence, call {call}")
        assert not bool((d_dev != 0).any()), "alpha = 0 gave a delta other than +-0"
        eff = ops.ntuple_promoted_weights(w_dev, pm, tuples, stages).cpu().numpy()
        assert not np.isnan(eff[ent]).any(), "an effective weight of a touched entry is NaN"
        assert not bool(acc.view(torch.int32).any())
    # alpha = 1/16: every partial sum exact
    adds = np.bincount(sref.entries(x0[keep], tuples, stages).ravel(), minlength=w.size)
    start = max(np.abs(w[~np.isnan(w)]).max(), np.abs(coh).max())
    assert 16 * start + adds.max() * 1 < 2 ** 24, (start, adds.max())  # in units of 1/16, |delta| <= 1/16
    w = _poisoned(_stage_weights(rng, tuples, stages, integer=True), np.zeros(n, np.uint8), tuples, stages)
    w_dev.copy_(torch.from_numpy(w))
    c_dev.copy_(torch.from_numpy(coh))
    pm.zero_()
    _race_call(ops, rule, dev, x0, k, w_dev, c_dev, acc, tuples, stages, pm, mk, d_dev, 0.0625)
    want_d = np.where(keep, k * np.float32(0.0625), np.float32(0)).astype(np.float32)
    np.testing.assert_array_equal(d_dev.cpu().numpy(), want_d)
    wp, want_m, cp = pref.promote(distinct, w, np.zeros(n, np.uint8), tuples, stages, None, coh if tc else None)
    if tc:
        _, e64, a64, _, _ = sref.tc_apply_f64(x0, want_d, wp, cp, tuples, stages, mask)
        de, da = e64 - cp[:, 0].astype(np.float64), a64 - cp[:, 1].astype(np.float64)  # exact: small multiples of 1/16
        want_w, want_c = sref.tc_apply_f32(de.astype(np.float32), da.astype(np.float32), wp, cp)
        _same_bits(c_dev.cpu().numpy(), want_c, "coherence")
    else:
        want_w = sref.td_apply_f64(x0, want_d, wp, tuples, stages, mask)[0].astype(np.float32)
        _same_bits(c_dev.cpu().numpy(), coh, "coherence")
    _same_bits(w_dev.cpu().numpy(), want_w, "weights")
    np.testing.assert_array_equal(pm.cpu().numpy(), want_m, "marks")
    assert not bool(acc.view(torch.int32).any())


@pytest.mark.gpu
def test_promotion_alone_keeps_every_effective_weight(ops, played):
    """alpha = 0 (delta 0 everywhere): the call only promotes; every effective weight and stage 0 stay bit for bit"""
    dev = _gpu()
    stages, tuples = CASES["s3"]
    rng = np.random.default_rng(300)
    n = nref.num_weights(tuples)
    w = torch.from_numpy(_stage_weights(rng, tuples, stages)).to(dev)
    pm = torch.zeros(n, dtype=torch.uint8, device=dev)
    eff0 = ops.ntuple_promoted_weights(w, pm, tuples, stages)
    w0 = w.clone()
    b = torch.from_numpy(played).to(dev)
    ops.ntuple_td_update(b, torch.zeros(b.shape[0], device=dev), w, tuples, alpha=0.0, stages=stages, promoted=pm)
    assert bool(pm.any())
    assert torch.equal(ops.ntuple_promoted_weights(w, pm, tuples, stages).view(torch.int32), eff0.view(torch.int32))
    assert torch.equal(w[:n], w0[:n])


@pytest.mark.gpu
def test_all_marks_and_one_stage_equal_the_staged_ops(ops, played):
    dev = _gpu()
    rng = np.random.default_rng(400)
    b = torch.from_numpy(played).to(dev)
    m = b.shape[0]
    target = torch.from_numpy(rng.integers(-64, 65, size=m).astype(np.float32)).to(dev)
    for stages, tuples in ((CASES["s3"]), ((), SMALL)):
        n = nref.num_weights(tuples)
        S = len(stages) + 1
        w = torch.from_numpy(_stage_weights(rng, tuples, stages, integer=True)).to(dev)
        full = torch.full((n,), (1 << (S - 1)) - 1 if S > 1 else 0x5A, dtype=torch.uint8, device=dev)
        pm = full.clone()
        for op in ("value", "greedy", "expectimax"):
            fn = getattr(ops, f"ntuple_{op}")
            bb = b[:200] if op == "expectimax" else b
            got, want = fn(bb, w, tuples, stages=stages, promoted=pm), fn(bb, w, tuples, stages=stages)
            if op == "value":
                got, want = {"v": got}, {"v": want}
            for k in got:
                assert torch.equal(got[k].view(torch.uint8), want[k].view(torch.uint8)), (stages, op, k)
        for rule in ("td0", "tc"):
            wa, wb = w.clone(), w.clone()
            ca, cb = torch.zeros((S * n, 2), device=dev), torch.zeros((S * n, 2), device=dev)
            acc = torch.zeros((S * n, 2), device=dev)
            if rule == "td0":
                da = ops.ntuple_td_update(b, target, wa, tuples, alpha=0.0625, stages=stages, promoted=pm)
                db = ops.ntuple_td_update(b, target, wb, tuples, alpha=0.0625, stages=stages)
            else:
                da = ops.ntuple_tc_update(b, target, wa, ca, acc, tuples, alpha=0.0625, stages=stages, promoted=pm)
                db = ops.ntuple_tc_update(b, target, wb, cb, acc, tuples, alpha=0.0625, stages=stages)
            assert torch.equal(da, db) and torch.equal(wa, wb) and torch.equal(ca, cb), (stages, rule)
        assert torch.equal(pm, full), "the marks changed"


@pytest.mark.gpu
def test_argument_errors(ops):
    dev = _gpu()
    stages, tuples = (4,), SMALL
    n = nref.num_weights(tuples)
    b = torch.zeros((8, 16), dtype=torch.uint8, device=dev)
    w = torch.ones(2 * n, device=dev)
    buf = torch.zeros(n + 8, dtype=torch.uint8, device=dev)
    for bad in (torch.zeros(n, dtype=torch.uint8), torch.zeros(n + 1, dtype=torch.uint8, device=dev),
                torch.zeros(n, dtype=torch.int8, device=dev), torch.zeros((n, 1), dtype=torch.uint8, device=dev),
                torch.zeros(2 * n, dtype=torch.uint8, device=dev)[::2], buf[1:n + 1], np.zeros(n, np.uint8)):
        for call in (lambda: ops.ntuple_value(b, w, tuples, stages=stages, promoted=bad),
                     lambda: ops.ntuple_greedy(b, w, tuples, stages=stages, promoted=bad),
                     lambda: ops.ntuple_td_update(b, torch.zeros(8, device=dev), w, tuples, alpha=0.1, stages=stages, promoted=bad)):
            with pytest.raises(ValueError):
                call()
    assert bool((w == 1).all())


# ---- CUDA graphs, the network, the learner and the policies -----------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc", "lambda_td", "lambda_tc"])
def test_graph_replay_equals_eager(ops, played, rule):
    """greedy + one update captured once, replayed over several steps from clear marks, against eager calls.  The marks
    carry over from step to step; every step starts from the same integer weights and zero coherence (beta = 1), so that
    every sum is exact and the order of the atomics cannot change a bit."""
    dev = _gpu()
    stages, tuples = CASES["s3"]
    rng = np.random.default_rng(500)
    m, h = 2048, 3
    n = nref.num_weights(tuples)
    N = sref.num_weights(tuples, stages)
    w_init = torch.from_numpy(_stage_weights(rng, tuples, stages, integer=True)).to(dev)
    state = {"w": w_init.clone(), "c": torch.zeros((N, 2), device=dev), "p": torch.zeros(n, dtype=torch.uint8, device=dev)}
    eager = {k: v.clone() for k, v in state.items()}
    acc = torch.zeros((N, 2), device=dev)
    s_board = torch.zeros((m, 16), dtype=torch.uint8, device=dev)
    s_prev = torch.zeros((m, 16), dtype=torch.uint8, device=dev)
    s_ring = torch.zeros((h + 1, m, 16), dtype=torch.uint8, device=dev)
    s_rew = torch.zeros((h + 1, m), device=dev)
    s_end = torch.zeros((h + 1, m), dtype=torch.uint8, device=dev)
    target = torch.zeros(m, device=dev)

    def step(st, board, prev, ring, rew, end, out, d):
        w, c, p = st["w"], st["c"], st["p"]
        g = ops.ntuple_greedy(board, w, tuples, action_dtype=torch.uint8, out=out, stages=stages, promoted=p)
        kw = dict(alpha=0.015625, delta_out=d, stages=stages, promoted=p)
        if rule == "lambda_td":
            ops.ntuple_td_lambda_update(ring, rew, end, 2, w, tuples, lam=0.5, **kw)
        elif rule == "lambda_tc":
            ops.ntuple_tc_lambda_update(ring, rew, end, 2, w, c, acc, tuples, lam=0.5, **kw)
        else:
            torch.add(g["reward"], g["value"], out=target)
            if rule == "td0":
                ops.ntuple_td_update(prev, target, w, tuples, **kw)
            else:
                ops.ntuple_tc_update(prev, target, w, c, acc, tuples, **kw)

    g_out = {"action": torch.zeros(m, dtype=torch.uint8, device=dev), "state": torch.zeros((m, 16), dtype=torch.uint8, device=dev),
             "reward": torch.zeros(m, device=dev), "value": torch.zeros(m, device=dev)}
    d_out = torch.zeros(m, device=dev)
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        step({k: v.clone() for k, v in state.items()}, s_board, s_prev, s_ring, s_rew, s_end,
             {k: v.clone() for k, v in g_out.items()}, d_out.clone())
    torch.cuda.current_stream().wait_stream(stream)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step(state, s_board, s_prev, s_ring, s_rew, s_end, g_out, d_out)
    for _ in range(4):
        s_board.copy_(torch.from_numpy(played[rng.integers(0, played.shape[0], size=m)]))
        s_prev.copy_(torch.from_numpy(played[rng.integers(0, played.shape[0], size=m)]))
        s_ring.copy_(torch.from_numpy(played[rng.integers(0, played.shape[0], size=(h + 1, m))]))
        s_rew.copy_(torch.from_numpy(rng.choice(np.array([0, 4, 8, 256], np.float32), size=(h + 1, m))))
        s_end.copy_(torch.from_numpy((rng.random((h + 1, m)) < 0.1).astype(np.uint8)))
        for st in (state, eager):
            st["w"].copy_(w_init)
            st["c"].zero_()
        inputs = [t.clone() for t in (s_board, s_prev, s_ring, s_rew, s_end)]
        marks_before = state["p"].clone()
        graph.replay()
        e_out = {k: torch.empty_like(v) for k, v in g_out.items()}
        d_e = torch.empty_like(d_out)
        step(eager, *inputs, e_out, d_e)
        torch.cuda.synchronize()
        for k in g_out:
            assert torch.equal(g_out[k].view(torch.uint8), e_out[k].view(torch.uint8)), k
        assert torch.equal(d_out.view(torch.int32), d_e.view(torch.int32))
        for k in state:
            assert torch.equal(state[k].view(torch.uint8), eager[k].view(torch.uint8)), k
        assert not torch.equal(state["p"], marks_before), "a step promoted nothing"
    assert not torch.equal(state["w"], w_init)


@pytest.mark.gpu
def test_learner_and_state_dict(ops):
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner

    dev = _gpu()
    with pytest.raises(ValueError):
        NTupleNetwork(device=dev, promotion=True)
    for rule, horizon in (("td0", 1), ("tc", 1), ("td0", 3)):
        net = NTupleNetwork(device=dev, stages=(4,), promotion=True)
        n = net.promoted.numel()
        assert n == nref.num_weights(net.tuples) and not bool(net.promoted.any())
        env = VecGame(4096, output="torch", sync_free=True, rng_mode="philox")
        learner = TDAfterstateLearner(env, net, rule=rule, horizon=horizon, lam=0.25)
        learner.reset(7)
        counts = []
        for i in range(2000):
            learner.step()
            if i % 500 == 499:
                counts.append(int((net.promoted != 0).sum()))
        torch.cuda.synchronize()
        assert counts[0] > 0 and counts == sorted(counts), (rule, counts)
        assert not bool((net.promoted & 0xFE).any()), "a bit above S - 2 was set"
        assert bool(torch.isfinite(net.weights).all())
        sd = net.state_dict()
        board = env.observations()[0].clone()
        v = net.value(board)
        # marks into a promoting net: copied
        same = NTupleNetwork(device=dev, stages=(4,), promotion=True)
        same.load_state_dict(sd)
        assert torch.equal(same.promoted, net.promoted) and torch.equal(same.weights, net.weights)
        assert torch.equal(same.value(board), v)
        # marks into a non-promoting staged net: the effective weights, coherence of unmarked entries zeroed
        plain = NTupleNetwork(device=dev, stages=(4,))
        plain.load_state_dict(sd)
        assert plain.promoted is None and torch.equal(plain.value(board), v)
        assert torch.equal(plain.weights, ops.ntuple_promoted_weights(net.weights, net.promoted, net.tuples, net.stages))
        if rule == "tc":
            unmarked = torch.cat([torch.zeros(n, dtype=torch.bool, device=dev), net.promoted == 0])
            assert not bool(plain.coherence[unmarked].any())
            assert torch.equal(plain.coherence[~unmarked], net.coherence[~unmarked])
        # a dict without marks into a promoting net: every mark set, the same values
        back = NTupleNetwork(device=dev, stages=(4,), promotion=True)
        back.load_state_dict(plain.state_dict())
        assert bool((back.promoted == 1).all()) and torch.equal(back.value(board), v)
        with pytest.raises(ValueError):
            NTupleNetwork(device=dev, stages=(5,), promotion=True).load_state_dict(sd)
        with pytest.raises(ValueError):
            NTupleNetwork(SMALL, device=dev, stages=(4,), promotion=True).load_state_dict(sd)


@pytest.mark.gpu
def test_policies_under_device_runner(ops):
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import ExpectimaxPolicy, GreedyPolicy, NTupleNetwork
    from ml2048_b200.runner import DeviceRunner

    dev = _gpu()
    net = NTupleNetwork(SMALL, device=dev, stages=(3, 5), promotion=True)
    net.weights.copy_(torch.randn(net.weights.numel(), device=dev) * 100)
    net.promoted.copy_(torch.randint(0, 4, net.promoted.shape, dtype=torch.uint8, device=dev))
    eff = ops.ntuple_promoted_weights(net.weights, net.promoted, net.tuples, net.stages)
    env = VecGame(512, "improved", two_prob=0.7, output="torch", sync_free=True)
    env.reset(1)
    for name, pol in (("greedy", GreedyPolicy(net, reward_fn="improved")),
                      ("expectimax1", ExpectimaxPolicy(net, depth=1, reward_fn="improved", two_prob=0.7))):
        runner = DeviceRunner(env, 512)
        seen = []
        runner.add_callback("prepared", lambda e, idx: seen.append(e.observations()[0].clone()))
        runner.add_callback("stepped", lambda e, res, actions, lp: seen.append(actions.clone()))
        for _ in range(4):
            runner.step_once(pol)
        for board, actions in zip(seen[0::2], seen[1::2]):
            if name == "greedy":
                want = ops.ntuple_greedy(board, eff, net.tuples, reward_fn="improved", stages=net.stages)["action"]
            else:
                want = ops.ntuple_expectimax(board, eff, net.tuples, depth=1, two_prob=0.7, reward_fn="improved",
                                             stages=net.stages)["action"]
            assert torch.equal(actions.to(dev), want), name
