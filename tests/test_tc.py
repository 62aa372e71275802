"""
Temporal coherence learning on the GPU (``ops.ntuple_tc_update``, ``NTupleNetwork.tc_update``, ``TDAfterstateLearner(...,
rule="tc")``) against the NumPy definition in tests/_tc_ref.py.

- Exact cases (games whose entries are pairwise disjoint): delta, weights, E and A bit-exact; zero and non-zero starting
  coherence (A >= |E|, and A = 0); with and without a mask; K = 1 / 4 / 16 with lengths 1..6; M = 1, 255, 257 and boards of a
  played environment; canary words around weights, coherence, accumulator and delta; the accumulator all zero bits after
  every call.
- Colliding games (M = 4096 and 2^18, early-game boards, > 1000 adds to one entry): delta bit-exact; weights, E and A within
  the float32 rounding bound of a float64 reference; untouched entries bit-identical; accumulator zero.
- Entries whose deltas are all +-0 do not change (-0 weights included); a NaN delta reaches only its own game's entries.
- CUDA-graph replay against eager over three replays.
- The learner with rule="tc": first step masked, finished games updated toward 0, delta = alpha * (y - v) bit for bit,
  state_dict round trips with and without coherence, a bad rule raises; from zero weights it beats the random policy.
"""

from __future__ import annotations

import time

import numpy as np
import pytest
import torch

import _ntuple_ref as nref
import _tc_ref as ref
from _ntuple_gpu import _gpu, ops  # noqa: F401 (ops is a fixture)

CANARY = 0x5A5A5A5A


def _guarded(shape, dtype, dev, fill=None, pad: int = 64):
    """a tensor inside a buffer of canary words, and a check that the canaries are intact"""
    count = int(np.prod(shape))
    nbytes = count * torch.empty(0, dtype=dtype).element_size()
    buf = torch.full((2 * pad + (nbytes + 3) // 4,), CANARY, dtype=torch.int32, device=dev)
    clean = buf.clone().view(torch.uint8)
    raw = buf.view(torch.uint8)
    body = raw[4 * pad:4 * pad + nbytes].view(dtype).view(shape)
    if fill is not None:
        body.copy_(fill)

    def intact():
        assert torch.equal(raw[:4 * pad], clean[:4 * pad]), "bytes before the buffer were written"
        assert torch.equal(raw[4 * pad + nbytes:], clean[4 * pad + nbytes:]), "bytes after the buffer were written"

    return body, intact


def _disjoint_rows(boards, tuples, want: int) -> np.ndarray:
    """indices of boards whose entry sets are pairwise disjoint (and without repeats inside one board)"""
    used, keep = set(), []
    for i, row in enumerate(nref.entries(boards, tuples)):
        s = set(int(x) for x in row)
        if len(s) == row.size and not (s & used):
            used |= s
            keep.append(i)
            if len(keep) == want:
                break
    return np.array(keep, np.int64)


def _played_boards(m: int, steps: int = 60) -> np.ndarray:
    from ml2048_b200 import VecGame

    env = VecGame(m, output="torch", rng_mode="philox")
    env.reset(11)
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    for _ in range(steps):
        env.prepare()
        env.step(torch.randint(0, 4, (m,), device="cuda", generator=g))
    return env.observations()[0].cpu().numpy().copy()


def _coherence(rng, n: int, kind: str) -> np.ndarray:
    if kind == "zero":
        return np.zeros((n, 2), np.float32)
    c = (rng.standard_normal((n, 2)) * 5).astype(np.float32)
    c[:, 1] = np.abs(c[:, 1]) + np.abs(c[:, 0])  # A >= |E|
    c[::5] = 0.0  # A = 0: beta = 1
    return c


def _same_bits(got: np.ndarray, want: np.ndarray) -> None:
    """bit-identical float32, except that a NaN matches any NaN"""
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan)
    np.testing.assert_array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))


def _zero_bits(acc: torch.Tensor) -> None:
    assert not bool(acc.view(torch.int32).any()), "the accumulator is not all zero bits"


# ---- exact cases --------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["k1", "k4", "k16"])
def test_tc_update_exact_cases(ops, shape):
    """k1 / k4: games whose entries are pairwise disjoint, random weights, one call after another on the same tensors.
    k16 has 1-cell tuples, so almost every pair of games shares an entry; there every call starts from small integer weights
    and targets with alpha = 1/16, so every delta is a multiple of 1/16 below 2^7 and every sum of them is exact in float32
    in any order: the atomics' order cannot change a bit."""
    dev = _gpu()
    rng = np.random.default_rng({"k1": 1, "k4": 2, "k16": 3}[shape])
    tuples = {"k1": ((3, 7, 11, 15, 14, 13),), "k4": nref.STANDARD_4X6,
              "k16": tuple(tuple(int(c) for c in rng.permutation(16)[:n]) for n in [1, 2, 3, 4, 5, 6, 2, 3, 4, 5, 1, 2, 3, 4, 5, 6])}[shape]
    n = nref.num_weights(tuples)
    dyadic = shape == "k16"
    uniform = rng.integers(0, 16, size=(20000, 16)).astype(np.uint8)  # few shared entries
    pool = np.concatenate([_played_boards(2048), uniform])
    rows = np.arange(257) + 1024 if dyadic else _disjoint_rows(pool, tuples, 257)
    assert rows.size == 257, rows.size
    alpha = 0.0625 if dyadic else 0.01
    for start in ("zero", "random"):
        w = (rng.standard_normal(n) * 100).astype(np.float32)
        c = _coherence(rng, n, start)
        w_dev, w_ok = _guarded((n,), torch.float32, dev, torch.from_numpy(w))
        c_dev, c_ok = _guarded((n, 2), torch.float32, dev, torch.from_numpy(c))
        a_dev, a_ok = _guarded((n, 2), torch.float32, dev, torch.zeros((n, 2)))
        for m in (1, 255, 257):
            b = pool[rows[:m]] if m != 255 else pool[rows[2:257]]
            y = (rng.standard_normal(m) * 200).astype(np.float32)
            for mask in (None, (rng.random(m) < 0.7).astype(np.uint8)):
                if dyadic:
                    w = rng.integers(-4, 5, n).astype(np.float32)
                    w_dev.copy_(torch.from_numpy(w))
                    y = rng.integers(-100, 101, m).astype(np.float32)
                d_dev, d_ok = _guarded((m,), torch.float32, dev)
                d = ops.ntuple_tc_update(torch.from_numpy(b).to(dev), torch.from_numpy(y).to(dev), w_dev, c_dev, a_dev, tuples,
                                         alpha=alpha, mask=None if mask is None else torch.from_numpy(mask).to(dev),
                                         delta_out=d_dev)
                assert d.data_ptr() == d_dev.data_ptr()
                want_d = ref.td_delta(b, y, w, tuples, alpha, mask)
                np.testing.assert_array_equal(d.cpu().numpy().view(np.uint32), want_d.view(np.uint32))
                w, c = ref.tc_apply_f32(*ref.tc_accumulate(b, want_d, tuples, mask), w, c)
                np.testing.assert_array_equal(w_dev.cpu().numpy().view(np.uint32), w.view(np.uint32))
                np.testing.assert_array_equal(c_dev.cpu().numpy().view(np.uint32), c.view(np.uint32))
                _zero_bits(a_dev)
                d_ok()
        w_ok()
        c_ok()
        a_ok()


# ---- colliding games ----------------------------------------------------------------------------------


def _tc_tolerance_check(w, c, w0, c0, w64, e64, a64, adds, sabs) -> None:
    touched = adds > 0
    for got, x0 in ((w, w0), (c[:, 0], c0[:, 0]), (c[:, 1], c0[:, 1])):
        np.testing.assert_array_equal(got[~touched].view(np.uint32), x0[~touched].view(np.uint32))
    beta = ref.tc_beta_f32(c0).astype(np.float64)[touched]
    u, k = 2.0 ** -24, adds[touched]
    # w: the k adds of dE, then beta's division, the product and the add each round once
    for got, want, bound in ((w, w64, (k + 2) * u * (np.abs(w0[touched].astype(np.float64)) + beta * sabs[touched])),
                             (c[:, 0], e64, k * u * (np.abs(c0[touched, 0].astype(np.float64)) + sabs[touched])),
                             (c[:, 1], a64, k * u * (np.abs(c0[touched, 1].astype(np.float64)) + sabs[touched]))):
        err = np.abs(got[touched].astype(np.float64) - want[touched])
        assert (err <= bound).all(), (err - bound).max()


@pytest.mark.gpu
@pytest.mark.parametrize("m", [4096, 1 << 18])
def test_tc_update_colliding_games(ops, m):
    """early-game boards (few tiles, small exponents): thousands of adds land on the same entries"""
    dev = _gpu()
    rng = np.random.default_rng(31)
    tuples = nref.STANDARD_4X6
    n = nref.num_weights(tuples)
    w0 = (rng.standard_normal(n) * 10).astype(np.float32)
    c0 = _coherence(rng, n, "random")
    b = np.where(rng.random((m, 16)) < 0.7, 0, rng.integers(1, 4, size=(m, 16))).astype(np.uint8)
    y = (rng.standard_normal(m) * 30).astype(np.float32)
    mask = (rng.random(m) < 0.8).astype(np.uint8)
    w_dev, w_ok = _guarded((n,), torch.float32, dev, torch.from_numpy(w0))
    c_dev, c_ok = _guarded((n, 2), torch.float32, dev, torch.from_numpy(c0))
    a_dev, a_ok = _guarded((n, 2), torch.float32, dev, torch.zeros((n, 2)))
    d_dev, d_ok = _guarded((m,), torch.float32, dev)
    d = ops.ntuple_tc_update(torch.from_numpy(b).to(dev), torch.from_numpy(y).to(dev), w_dev, c_dev, a_dev, tuples, alpha=0.003,
                             mask=torch.from_numpy(mask).to(dev), delta_out=d_dev)
    want_d = ref.td_delta(b, y, w0, tuples, 0.003, mask)
    np.testing.assert_array_equal(d.cpu().numpy().view(np.uint32), want_d.view(np.uint32))
    w64, e64, a64, adds, sabs = ref.tc_apply_f64(b, want_d, w0, c0, tuples, mask)
    assert adds.max() > 1000
    _tc_tolerance_check(w_dev.cpu().numpy(), c_dev.cpu().numpy(), w0, c0, w64, e64, a64, adds, sabs)
    _zero_bits(a_dev)
    for ok in (w_ok, c_ok, a_ok, d_ok):
        ok()


@pytest.mark.gpu
def test_tc_update_zero_deltas_and_nan(ops):
    """alpha = 0 gives every game a delta of +-0: nothing changes, -0 weights included.  A NaN target in one game makes NaN
    exactly the entries of that game."""
    dev = _gpu()
    rng = np.random.default_rng(32)
    tuples = ((0, 1, 2), (4, 5), (0, 4, 8, 12))
    n = nref.num_weights(tuples)
    b = _played_boards(4096)
    w0 = (rng.standard_normal(n) * 10).astype(np.float32)
    w0[::2] = -0.0
    c0 = _coherence(rng, n, "random")
    w_dev, c_dev = torch.from_numpy(w0).to(dev), torch.from_numpy(c0).to(dev)
    acc = torch.zeros((n, 2), device=dev)
    bd = torch.from_numpy(b).to(dev)
    y = torch.from_numpy((rng.standard_normal(b.shape[0]) * 100).astype(np.float32)).to(dev)
    d = ops.ntuple_tc_update(bd, y, w_dev, c_dev, acc, tuples, alpha=0.0)
    assert bool((d == 0).all()) and bool((torch.signbit(d)).any()) and bool((~torch.signbit(d)).any())
    assert torch.equal(w_dev.view(torch.int32), torch.from_numpy(w0).to(dev).view(torch.int32))
    assert torch.equal(c_dev.view(torch.int32), torch.from_numpy(c0).to(dev).view(torch.int32))
    _zero_bits(acc)
    # a NaN delta: game 17's entries only
    y[17] = float("nan")
    ops.ntuple_tc_update(bd, y, w_dev, c_dev, acc, tuples, alpha=0.001)
    mine = np.zeros(n, bool)
    mine[nref.entries(b[17:18], tuples).ravel()] = True
    w, c = w_dev.cpu().numpy(), c_dev.cpu().numpy()
    assert np.isnan(w[mine]).all() and np.isnan(c[mine]).all()
    assert np.isfinite(w[~mine]).all() and np.isfinite(c[~mine]).all()
    _zero_bits(acc)


# ---- CUDA graphs --------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_graph_replay_equals_eager(ops):
    dev = _gpu()
    rng = np.random.default_rng(40)
    tuples = nref.STANDARD_4X6
    n = nref.num_weights(tuples)
    m = 70001
    w = torch.from_numpy((rng.standard_normal(n) * 10).astype(np.float32)).to(dev)
    coh = torch.from_numpy(_coherence(rng, n, "random")).to(dev)
    acc = torch.zeros((n, 2), device=dev)
    static_b = torch.zeros((m, 16), dtype=torch.uint8, device=dev)
    static_y = torch.zeros((m,), dtype=torch.float32, device=dev)
    d_out = torch.empty((m,), dtype=torch.float32, device=dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ops.ntuple_tc_update(static_b, static_y, w, coh, acc, tuples, alpha=0.002, delta_out=d_out)
    played = _played_boards(m, 30)
    for rep in range(3):
        b = torch.from_numpy(played if rep == 0 else rng.integers(0, 6, size=(m, 16)).astype(np.uint8)).to(dev)
        y = torch.randn(m, device=dev) * 20
        static_b.copy_(b)
        static_y.copy_(y)
        w0, c0 = w.clone(), coh.clone()
        graph.replay()
        w_r, c_r = w.clone(), coh.clone()
        _zero_bits(acc)
        w_e, c_e = w0.clone(), c0.clone()
        d = ops.ntuple_tc_update(b, y, w_e, c_e, acc, tuples, alpha=0.002)
        _zero_bits(acc)
        assert torch.equal(d_out.view(torch.int32), d.view(torch.int32))
        bh, dh, w0h, c0h = b.cpu().numpy(), d.cpu().numpy(), w0.cpu().numpy(), c0.cpu().numpy()
        want = ref.tc_apply_f64(bh, dh, w0h, c0h, tuples)
        _tc_tolerance_check(w_r.cpu().numpy(), c_r.cpu().numpy(), w0h, c0h, *want)
        _tc_tolerance_check(w_e.cpu().numpy(), c_e.cpu().numpy(), w0h, c0h, *want)


# ---- the network class and the learner ------------------------------------------------------------------


@pytest.mark.gpu
def test_network_tc_state_dict(ops):
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner

    dev = _gpu()
    tuples = ((0, 1, 2), (4, 5))
    net = NTupleNetwork(tuples, device=dev)
    assert net.coherence is None and "coherence" not in net.state_dict()
    b = torch.from_numpy(_played_boards(512)).to(dev)
    net.tc_update(b, torch.randn(512, device=dev) * 10, 0.01)
    assert tuple(net.coherence.shape) == (net.weights.numel(), 2) and bool(net.coherence.any())
    state = net.state_dict()
    assert torch.equal(state["coherence"], net.coherence) and state["coherence"].data_ptr() != net.coherence.data_ptr()
    other = NTupleNetwork(tuples, device=dev)
    other.load_state_dict(state)
    assert torch.equal(other.weights, net.weights) and torch.equal(other.coherence, net.coherence)
    # the same update continues the same way from the loaded state
    y = torch.randn(512, device=dev) * 10
    d1 = net.tc_update(b, y, 0.01)
    d2 = other.tc_update(b, y, 0.01)
    assert torch.equal(d1, d2)
    # an older dict without coherence loads, and drops the coherence state
    old = {"tuples": state["tuples"], "weights": state["weights"]}
    other.load_state_dict(old)
    assert other.coherence is None and torch.equal(other.weights, state["weights"])
    for bad in (state["coherence"][:-1], state["coherence"].double(), state["coherence"].reshape(-1)):
        with pytest.raises(ValueError):
            other.load_state_dict(dict(state, coherence=bad))
    with pytest.raises(ValueError):
        TDAfterstateLearner(VecGame(64, output="torch", sync_free=True), net, rule="bogus")


@pytest.mark.gpu
def test_learner_tc_first_step_masks_and_terminal_targets(ops):
    """the first step after reset() updates nothing; a game that ended is updated toward 0; delta = alpha * (y - v)"""
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner, default_tc_alpha

    dev = _gpu()
    net = NTupleNetwork(device=dev)
    env = VecGame(4096, output="torch", sync_free=True)
    learner = TDAfterstateLearner(env, net, rule="tc")
    assert learner.alpha == default_tc_alpha(4096)
    learner = TDAfterstateLearner(env, net, alpha=0.01, rule="tc")
    learner.reset(3)
    learner.step()
    assert not bool(net.weights.any()) and not bool(learner.delta.any()) and not bool(net.coherence.any())
    ended = 0
    for _ in range(300):
        prev_after = learner._prev_after.clone()
        prev_ended = learner._prev_ended.clone()
        w = net.weights.clone()
        learner.step()
        v = ops.ntuple_value(prev_after, w, net.tuples)
        y = torch.where(prev_ended, torch.zeros_like(v), learner._out["reward"] + learner._out["value"])
        want = torch.tensor(0.01, dtype=torch.float32, device=dev) * (y - v)
        assert torch.equal(learner.delta.view(torch.int32), want.view(torch.int32))
        ended += int(prev_ended.sum())
    assert ended > 0
    _zero_bits(net._tc_accum)


@pytest.mark.gpu
def test_learner_tc_beats_the_random_policy(ops):
    """TC afterstate learning from zero weights, M = 2^14 games, the standard 4x6 network, the default TC alpha, a fixed
    number of steps (100 000 steps, 13.2 s on one B200 at 1000 W).  The random policy (tests/golden/random_policy_stats.npz):
    mean score 1 015, 512 reached in 0.014 % of episodes.

    Measured on that B200 over the 364 826 episodes that end in the last quarter of the run: mean score 21 894, 512 reached
    in 98.8 %, 1024 in 87.8 %, 2048 in 43.1 %.  The thresholds are about half of the score and of the 512 share."""
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner

    dev = _gpu()
    net = NTupleNetwork(device=dev)
    env = VecGame(1 << 14, output="torch", sync_free=True, rng_mode="philox")
    learner = TDAfterstateLearner(env, net, rule="tc")
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
    print(f"tc learner: {steps} steps in {elapsed:.1f} s, {eps} episodes in the last quarter, mean score {mean_score:.0f}, "
          f">= 512: {share512:.3f}, >= 1024: {hist[10:].sum() / max(eps, 1):.3f}, >= 2048: {hist[11:].sum() / max(eps, 1):.4f}")
    assert eps > 100
    assert mean_score > THRESHOLDS["mean_score"], mean_score
    assert share512 > THRESHOLDS["share512"], share512


LEARN_STEPS = 100000
THRESHOLDS = {"mean_score": 11000.0, "share512": 0.5}
