"""
Delayed TD(lambda) / TC(lambda) on the GPU (``ops.ntuple_td_lambda_update`` / ``ntuple_tc_lambda_update``,
``NTupleNetwork.td_lambda_update`` / ``tc_lambda_update``, ``TDAfterstateLearner(..., horizon=h, lam=...)``) against the NumPy
definition in tests/_lambda_ref.py.

- Exact cases, both rules: delta bit for bit for K = 1 / 4 / 16, M = 1, 255, 257, h = 1, 3, 16, every newest slot, ends inside
  the windows, with and without a mask; weights (and E / A for TC) bit for bit where x_0's entries are pairwise disjoint
  (K = 1 / 4) or where every sum is exact in any order (K = 16, dyadic values); canary words around every buffer.
- h = 16 at M = 2^23 + 5, where the after ring passes 2^31 bytes, both rules and once with stages: x_0 in the first and in
  the last slot, a mask of rows at both ends and a seeded sample; delta bit for bit there and 0 elsewhere, the weights
  within the float32 bound of the float64 reference over the sampled rows.
- h = 1 equals ntuple_td_update and ntuple_tc_update on colliding games: delta, weights and coherence bit for bit.
- CUDA-graph replay against eager, both rules.
- The learner with horizon=3, both rules: the first 3 steps after reset() update nothing; each later delta equals the
  reference from the ring and a weights snapshot taken before the step; games that ended are truncated; bad horizon / lam
  raise.  From zero weights it beats the random policy.
"""

from __future__ import annotations

import time

import numpy as np
import pytest
import torch

import _lambda_ref as ref
import _ntuple_ref as nref
import _stage_ref as sref
import _tc_ref as tref
from _ntuple_gpu import _gpu, ops  # noqa: F401 (ops is a fixture)
from test_tc import _coherence, _disjoint_rows, _guarded, _played_boards, _same_bits, _zero_bits


def _update(ops, rule, rings, newest, w_dev, c_dev, a_dev, tuples, **kw):
    if rule == "tc":
        return ops.ntuple_tc_lambda_update(*rings, newest, w_dev, c_dev, a_dev, tuples, **kw)
    return ops.ntuple_td_lambda_update(*rings, newest, w_dev, tuples, **kw)


def _want_update(rule, x0, d, w, c, tuples, mask):
    if rule == "tc":
        return tref.tc_apply_f32(*tref.tc_accumulate(x0, d, tuples, mask), w, c)
    return nref.td_apply_f32(x0, d, w, tuples, mask), c


# ---- exact cases --------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc"])
@pytest.mark.parametrize("shape", ["k1", "k4", "k16"])
def test_lambda_update_exact_cases(ops, shape, rule):
    """k1 / k4: x_0 of the games have pairwise disjoint entries, random weights and values.  k16 has 1-cell tuples, so the
    games share entries; there the weights are small integers, the rewards 0..16, alpha = 1/16 and lambda 0 or 1, so every
    return is an integer, every delta a multiple of 1/16 and every sum of them exact in any order."""
    dev = _gpu()
    rng = np.random.default_rng({"k1": 11, "k4": 12, "k16": 13}[shape] + (rule == "tc"))
    tuples = {"k1": ((3, 7, 11, 15, 14, 13),), "k4": nref.STANDARD_4X6,
              "k16": tuple(tuple(int(c) for c in rng.permutation(16)[:n]) for n in [1, 2, 3, 4, 5, 6, 2, 3, 4, 5, 1, 2, 3, 4, 5, 6])}[shape]
    n = nref.num_weights(tuples)
    dyadic = shape == "k16"
    uniform = rng.integers(0, 16, size=(20000, 16)).astype(np.uint8)
    pool = np.concatenate([_played_boards(2048), uniform])
    rows = np.arange(257) + 1024 if dyadic else _disjoint_rows(pool, tuples, 257)
    assert rows.size == 257, rows.size
    alpha = 0.0625 if dyadic else 0.01
    w = (rng.standard_normal(n) * 100).astype(np.float32)
    c = _coherence(rng, n, "random")
    w_dev, w_ok = _guarded((n,), torch.float32, dev, torch.from_numpy(w))
    c_dev, c_ok = _guarded((n, 2), torch.float32, dev, torch.from_numpy(c))
    a_dev, a_ok = _guarded((n, 2), torch.float32, dev, torch.zeros((n, 2)))
    calls = 0
    for h in (1, 3, 16):
        for m in (1, 255, 257):
            newest = int(rng.integers(0, h + 1))
            after = pool[rng.integers(0, pool.shape[0], size=(h + 1, m))]
            after[(newest + 1) % (h + 1)] = pool[rows[:m]] if m != 255 else pool[rows[2:257]]  # x_0
            reward = rng.choice(np.array([0, 4, 8, 16] if dyadic else [0, 4, 8, 16, 256, 2048], np.float32), size=(h + 1, m))
            ended = (rng.random((h + 1, m)) < 0.15).astype(np.uint8)
            for mask in (None, (rng.random(m) < 0.7).astype(np.uint8)):
                lam = float(calls % 2) if dyadic else (0.5, 0.37)[calls % 2]
                calls += 1
                if dyadic:
                    w = rng.integers(-4, 5, n).astype(np.float32)
                    w_dev.copy_(torch.from_numpy(w))
                rings, oks = [], []
                for arr, dt in ((after, torch.uint8), (reward, torch.float32), (ended, torch.uint8)):
                    t, ok = _guarded(arr.shape, dt, dev, torch.from_numpy(arr))
                    rings.append(t)
                    oks.append(ok)
                d_dev, d_ok = _guarded((m,), torch.float32, dev)
                d = _update(ops, rule, rings, newest, w_dev, c_dev, a_dev, tuples, alpha=alpha, lam=lam,
                            mask=None if mask is None else torch.from_numpy(mask).to(dev), delta_out=d_dev)
                assert d.data_ptr() == d_dev.data_ptr()
                want_d, x0 = ref.ring_delta(after, reward, ended, newest, w, tuples, lam, alpha, mask)
                _same_bits(d.cpu().numpy(), want_d)
                w, c = _want_update(rule, x0, want_d, w, c, tuples, mask)
                np.testing.assert_array_equal(w_dev.cpu().numpy().view(np.uint32), w.view(np.uint32))
                np.testing.assert_array_equal(c_dev.cpu().numpy().view(np.uint32), c.view(np.uint32))
                _zero_bits(a_dev)
                for ok in oks + [d_ok]:
                    ok()
                # the ring is input only
                for t, arr in zip(rings, (after, reward, ended)):
                    np.testing.assert_array_equal(t.cpu().numpy(), arr)
    w_ok()
    c_ok()
    a_ok()


@pytest.mark.gpu
@pytest.mark.parametrize("rule,stages", [("td0", ()), ("tc", ()), ("tc", (3, 5))])
def test_lambda_update_beyond_2gib_of_ring(ops, rule, stages):
    """h = 16, M = 2^23 + 5: the after ring is (17, M, 16) bytes, 2.28 GB, so the byte offsets of slots 8 and up pass 2^31.
    newest = 16 (x_0 in slot 0, x_h in the last slot) and newest = 15 (x_0 in the last slot).  The mask selects rows at both
    ends of M and a seeded sample: delta is 0 everywhere else (checked on the device), bit for bit the reference's on the
    selected rows, and the weights (and E / A) within the float32 bound of the float64 reference over those rows alone.
    0.5-0.8 s per case on one B200 (power limit not recorded)."""
    from test_ntuple import _td_tolerance_check
    from test_stages import SMALL
    from test_tc import _tc_tolerance_check

    dev = _gpu()
    h, m, lam, alpha = 16, (1 << 23) + 5, 0.5, 0.01
    tuples = SMALL
    n = sref.num_weights(tuples, stages)
    rng = np.random.default_rng(50 + len(stages) + (rule == "tc"))
    g = torch.Generator(device=dev)
    g.manual_seed(51)
    after = torch.randint(0, 18, (h + 1, m, 16), dtype=torch.uint8, device=dev, generator=g)
    table = torch.tensor([0.0, 4.0, 8.0, 256.0], device=dev)
    reward = table[torch.randint(0, 4, (h + 1, m), device=dev, generator=g)]
    ended = (torch.rand((h + 1, m), device=dev, generator=g) < 0.05).to(torch.uint8)
    rows = np.unique(np.concatenate([np.arange(256), np.arange(m - 256, m), rng.integers(0, m, 8192)]))
    r_dev = torch.from_numpy(rows).to(dev)
    mask = torch.zeros(m, dtype=torch.uint8, device=dev)
    mask[r_dev] = 1
    rings = (after[:, r_dev].cpu().numpy(), reward[:, r_dev].cpu().numpy(), ended[:, r_dev].cpu().numpy())
    w = (rng.standard_normal(n) * 10).astype(np.float32)
    c = _coherence(rng, n, "random")
    for newest in (16, 15):
        w_dev, c_dev = torch.from_numpy(w).to(dev), torch.from_numpy(c).to(dev)
        acc = torch.zeros((n, 2), device=dev)
        d = _update(ops, rule, (after, reward, ended), newest, w_dev, c_dev, acc, tuples, alpha=alpha, lam=lam, mask=mask,
                    stages=stages)
        assert not bool(d[mask == 0].any()), "a masked-out game has a delta"
        want_d, x0 = sref.ring_delta(*rings, newest, w, tuples, stages, lam, alpha)
        np.testing.assert_array_equal(x0, after[(newest + 1) % (h + 1)][r_dev].cpu().numpy())
        _same_bits(d[r_dev].cpu().numpy(), want_d)
        if rule == "tc":
            w64, e64, a64, adds, sabs = sref.tc_apply_f64(x0, want_d, w, c, tuples, stages)
            _tc_tolerance_check(w_dev.cpu().numpy(), c_dev.cpu().numpy(), w, c, w64, e64, a64, adds, sabs)
            _zero_bits(acc)
        else:
            w64, adds, sabs = sref.td_apply_f64(x0, want_d, w, tuples, stages)
            _td_tolerance_check(w_dev.cpu().numpy(), w, w64, adds, sabs)
            assert torch.equal(c_dev.cpu(), torch.from_numpy(c))
        assert adds.any()
    del after, reward, ended, mask, d
    torch.cuda.empty_cache()


# ---- h = 1 is TD(0) / TC ------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc"])
def test_h1_equals_td0_and_tc(ops, rule):
    """h = 1 against ntuple_td_update / ntuple_tc_update toward reward + V(x_1), 0 where x_0's game ended, on 4096 played
    boards that collide; integer weights and rewards and alpha = 1/16 keep every atomic sum exact, so the bits must agree"""
    dev = _gpu()
    rng = np.random.default_rng(21)
    tuples = nref.STANDARD_4X6
    n = nref.num_weights(tuples)
    m = 4096
    boards = _played_boards(2 * m, 40)
    w0 = torch.from_numpy(rng.integers(-4, 5, n).astype(np.float32)).to(dev)
    c0 = torch.from_numpy(_coherence(rng, n, "random")).to(dev)
    for newest in (0, 1):
        after = torch.from_numpy(boards.reshape(2, m, 16)).to(dev)
        reward = torch.from_numpy(rng.choice(np.array([0, 4, 8, 16], np.float32), size=(2, m))).to(dev)
        ended = torch.from_numpy((rng.random((2, m)) < 0.2).astype(np.uint8)).to(dev)
        mask = torch.from_numpy((rng.random(m) < 0.9).astype(np.uint8)).to(dev)
        old = 1 - newest
        target = torch.add(reward[newest], ops.ntuple_value(after[newest], w0, tuples)).masked_fill_(ended[old].bool(), 0.0)
        acc = torch.zeros((n, 2), device=dev)
        for lam in (0.0, 0.5, 1.0):  # h = 1 does not use lambda
            w_l, w_t, c_l, c_t = w0.clone(), w0.clone(), c0.clone(), c0.clone()
            if rule == "tc":
                d_l = ops.ntuple_tc_lambda_update(after, reward, ended, newest, w_l, c_l, acc, tuples, alpha=0.0625, lam=lam, mask=mask)
                d_t = ops.ntuple_tc_update(after[old], target, w_t, c_t, acc, tuples, alpha=0.0625, mask=mask)
            else:
                d_l = ops.ntuple_td_lambda_update(after, reward, ended, newest, w_l, tuples, alpha=0.0625, lam=lam, mask=mask)
                d_t = ops.ntuple_td_update(after[old], target, w_t, tuples, alpha=0.0625, mask=mask)
            assert torch.equal(d_l.view(torch.int32), d_t.view(torch.int32))
            assert torch.equal(w_l.view(torch.int32), w_t.view(torch.int32))
            assert torch.equal(c_l.view(torch.int32), c_t.view(torch.int32))
            _zero_bits(acc)
        assert bool((w_l != w0).any())


# ---- CUDA graphs --------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc"])
def test_graph_replay_equals_eager(ops, rule):
    """three replays on new ring contents (x_0 with pairwise disjoint entries, so the weights are exact) against eager calls
    from the same starting weights"""
    dev = _gpu()
    rng = np.random.default_rng(40)
    tuples = nref.STANDARD_4X6
    n = nref.num_weights(tuples)
    h, newest = 4, 2
    pool = np.concatenate([_played_boards(2048), rng.integers(0, 16, size=(40000, 16)).astype(np.uint8)])
    rows = _disjoint_rows(pool, tuples, 1000)
    m = rows.size
    assert m > 500, m
    w = torch.from_numpy((rng.standard_normal(n) * 10).astype(np.float32)).to(dev)
    coh = torch.from_numpy(_coherence(rng, n, "random")).to(dev)
    acc = torch.zeros((n, 2), device=dev)
    s_after = torch.zeros((h + 1, m, 16), dtype=torch.uint8, device=dev)
    s_reward = torch.zeros((h + 1, m), device=dev)
    s_ended = torch.zeros((h + 1, m), dtype=torch.uint8, device=dev)
    d_out = torch.empty((m,), device=dev)
    rings = (s_after, s_reward, s_ended)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _update(ops, rule, rings, newest, w, coh, acc, tuples, alpha=0.002, lam=0.7, delta_out=d_out)
    for rep in range(3):
        after = pool[rng.integers(0, pool.shape[0], size=(h + 1, m))]
        after[(newest + 1) % (h + 1)] = pool[rng.permutation(rows)]
        s_after.copy_(torch.from_numpy(after))
        s_reward.copy_(torch.from_numpy(rng.choice(np.array([0, 4, 8, 256], np.float32), size=(h + 1, m))))
        s_ended.copy_(torch.from_numpy((rng.random((h + 1, m)) < 0.1).astype(np.uint8)))
        w0, c0 = w.clone(), coh.clone()
        graph.replay()
        w_e, c_e = w0.clone(), c0.clone()
        d = _update(ops, rule, tuple(t.clone() for t in rings), newest, w_e, c_e, acc, tuples, alpha=0.002, lam=0.7)
        _zero_bits(acc)
        assert torch.equal(d_out.view(torch.int32), d.view(torch.int32))
        assert torch.equal(w.view(torch.int32), w_e.view(torch.int32)) and not torch.equal(w, w0)
        assert torch.equal(coh.view(torch.int32), c_e.view(torch.int32))
        want_d, _ = ref.ring_delta(after, s_reward.cpu().numpy(), s_ended.cpu().numpy(), newest, w0.cpu().numpy(), tuples, 0.7, 0.002)
        _same_bits(d.cpu().numpy(), want_d)


# ---- the network class and the learner ------------------------------------------------------------------


@pytest.mark.gpu
def test_learner_argument_errors(ops):
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner

    net = NTupleNetwork(((0, 1), (2,)), device=_gpu())
    env = VecGame(64, output="torch", sync_free=True)
    for bad in (0, 17, -1, True, 2.0, "3"):
        with pytest.raises(ValueError, match="horizon"):
            TDAfterstateLearner(env, net, horizon=bad)
    for bad in (-0.1, 1.5, float("nan"), True, "0.5", None):
        with pytest.raises(ValueError, match="lam"):
            TDAfterstateLearner(env, net, horizon=2, lam=bad)
    assert TDAfterstateLearner(env, net, horizon=16, lam=1).lam == 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc"])
def test_learner_horizon3(ops, rule):
    """the first 3 steps after reset() update nothing; from then on delta is the reference's from the ring and the weights
    before the step, bit for bit; windows with an end in them occur, and reset() empties the window again"""
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import DEFAULT_TC_LAMBDA_ALPHA_TIMES_GAMES, NTupleNetwork, TDAfterstateLearner, default_alpha

    dev = _gpu()
    h, lam, m = 3, 0.5, 4096
    net = NTupleNetwork(device=dev)
    env = VecGame(m, output="torch", sync_free=True)
    learner = TDAfterstateLearner(env, net, rule=rule, horizon=h)
    assert learner.alpha == (DEFAULT_TC_LAMBDA_ALPHA_TIMES_GAMES / m if rule == "tc" else default_alpha(m)) and learner.lam == 0.5
    learner = TDAfterstateLearner(env, net, alpha=1e-4, rule=rule, horizon=h, lam=lam)
    learner.reset(3)
    for _ in range(h):
        learner.step()
        assert not bool(net.weights.any()) and not bool(learner.delta.any())
        assert net.coherence is None or not bool(net.coherence.any())
    truncated = 0
    for t in range(h, 300):
        w = net.weights.clone()
        learner.step()
        newest = t % (h + 1)
        v = torch.stack([ops.ntuple_value(learner._after_ring[s], w, net.tuples) for s in range(h + 1)]).cpu().numpy()
        rho, ended = learner._reward_ring.cpu().numpy(), learner._ended_ring.cpu().numpy()
        want = ref.lambda_delta(ref.window(v, newest), ref.window(rho, newest), ref.window(ended, newest), lam, 1e-4)
        _same_bits(learner.delta.cpu().numpy(), want)
        truncated += int(ref.window(ended, newest)[:h].any(axis=0).sum())
    assert truncated > 0
    assert bool(net.weights.any()) and bool(torch.isfinite(net.weights).all())
    if rule == "tc":
        _zero_bits(net._tc_accum)
    learner.reset(4)
    w = net.weights.clone()
    for _ in range(h):
        learner.step()
        assert torch.equal(net.weights.view(torch.int32), w.view(torch.int32)) and not bool(learner.delta.any())
    learner.step()
    assert not torch.equal(net.weights, w)


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc"])
def test_learner_lambda_beats_the_random_policy(ops, rule):
    """delayed TD(lambda) / TC(lambda) afterstate learning from zero weights at each rule's best setting of
    tools/lambda_bench.py (TD: h = 3, lambda = 0.25; TC: h = 2, lambda = 0.25), M = 2^14 games, the standard 4x6 network, the
    default alpha, 100 000 steps.  The random policy (tests/golden/random_policy_stats.npz): mean score 1 015, 512 reached in
    0.014 % of episodes.

    Measured on one B200 at 1000 W over the episodes that end in the last quarter of the run: TD mean score 22 177, 512
    reached in 98.3 % (7.0 s); TC 19 661 and 98.5 % (12.1 s).  The thresholds are about half of the score and of the 512
    share."""
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner

    dev = _gpu()
    net = NTupleNetwork(device=dev)
    env = VecGame(1 << 14, output="torch", sync_free=True, rng_mode="philox")
    learner = TDAfterstateLearner(env, net, rule=rule, horizon=3 if rule == "td0" else 2, lam=0.25)
    learner.reset(7)
    t0 = time.perf_counter()
    steps = LEARN_STEPS
    for i in range(steps):
        if i == 3 * steps // 4:
            env.episode_stats(reset=True)
        learner.step()
    st = env.episode_stats()
    elapsed = time.perf_counter() - t0
    eps = st["episodes"]
    hist = np.asarray(st["max_tile_hist"], np.int64)
    mean_score = st["score_sum"] / max(eps, 1)
    share512 = hist[9:].sum() / max(eps, 1)
    print(f"{rule} lambda learner: {steps} steps in {elapsed:.1f} s, {eps} episodes in the last quarter, mean score "
          f"{mean_score:.0f}, >= 512: {share512:.3f}, >= 1024: {hist[10:].sum() / max(eps, 1):.3f}, "
          f">= 2048: {hist[11:].sum() / max(eps, 1):.4f}")
    assert eps > 100
    assert mean_score > THRESHOLDS[rule]["mean_score"], mean_score
    assert share512 > THRESHOLDS[rule]["share512"], share512


LEARN_STEPS = 100000
THRESHOLDS = {"td0": {"mean_score": 11000.0, "share512": 0.5}, "tc": {"mean_score": 10000.0, "share512": 0.5}}
