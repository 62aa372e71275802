"""
Expectimax over an n-tuple network on the GPU (``ops.ntuple_expectimax``, ``NTupleNetwork.expectimax``, ``ExpectimaxPolicy``)
against the NumPy definition in tests/_expectimax_ref.py, which takes ``ops.afterstates`` as its move function.

- Bit-exact action, state, reward, value and q.  Depth 1: every combination of the four reward kinds, two_prob 0 / 0.3 /
  0.8 / 1, random / zero / NaN-and-inf weights and K = 1 / 4 / 16 tuples, at M = 1, 255, 257 and on boards from a played
  environment; M = 2^20 + 3 on sampled rows.  Depth 2: each of those values at least once.  uint8 and int64 actions, canary
  words around every output.
- CUDA-graph replay equals eager bit for bit.
- ``ExpectimaxPolicy`` under ``DeviceRunner`` plays what ``ops.ntuple_expectimax`` chooses.
- Strength: on one trained network, depth-1 expectimax scores more than the greedy move over the same games.
"""

from __future__ import annotations

import time

import numpy as np
import pytest
import torch

import _expectimax_ref as xref
import _ntuple_ref as ref
from _ntuple_gpu import _gpu, ops  # noqa: F401 (ops is a fixture)

KINDS = ("normal", "improved", "rank", "maxcell")
TWO_PROBS = (0.0, 0.3, 0.8, 1.0)
CANARY = 0x5A5A5A5A


def _played_boards(m: int, steps: int, seed: int) -> np.ndarray:
    from ml2048_b200 import VecGame

    env = VecGame(m, output="torch", rng_mode="philox")
    env.reset(seed)
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    for _ in range(steps):
        env.prepare()
        env.step(torch.randint(0, 4, (m,), device="cuda", generator=g))
    return env.observations()[0].cpu().numpy().copy()


def _random_boards(rng, m: int, empty_share: float) -> np.ndarray:
    """exponents 1..17 (15, 16 and 17 among them) with a share of empty cells, small exponents (ties) in every third board"""
    b = np.where(rng.random((m, 16)) < empty_share, 0, rng.integers(1, 18, size=(m, 16))).astype(np.uint8)
    b[::3] = np.where(rng.random(b[::3].shape) < empty_share, 0, rng.integers(1, 3, size=b[::3].shape))
    return b


DEAD = np.tile(np.array([1, 2, 1, 2, 2, 1, 2, 1], np.uint8), 2)
ONE_TILE = np.array([3] + [0] * 15, np.uint8)          # 15 empty cells after a move
ONE_EMPTY = np.array(list(range(1, 16)) + [0], np.uint8)  # one empty cell after a move


def _pool(rng, n_random: int, played: np.ndarray, empty_share: float) -> np.ndarray:
    pool = np.concatenate([np.stack([ONE_TILE, DEAD, ONE_EMPTY]), _random_boards(rng, n_random, empty_share), played])
    pool[1::41] = DEAD
    return pool


def _tuples(rng, shape: str):
    return {"k1": ((3, 7, 11, 15, 14, 13),), "k4": ref.STANDARD_4X6,
            "k16": tuple(tuple(int(c) for c in rng.permutation(16)[:n]) for n in (1, 2, 3, 4, 5, 2, 3, 4, 5, 1, 2, 3, 4, 5, 3, 2))}[shape]


def _weights(rng, tuples, kind: str) -> np.ndarray:
    n = ref.num_weights(tuples)
    if kind == "zero":
        return np.zeros(n, np.float32)
    w = (rng.standard_normal(n) * 100).astype(np.float32)
    if kind == "naninf":
        w[rng.random(n) < 0.02] = np.nan
        w[rng.random(n) < 0.01] = -np.inf
        w[rng.random(n) < 0.005] = np.inf
    return w


def _move(ops, kind):
    def move(boards: np.ndarray):
        a = ops.afterstates(torch.from_numpy(np.ascontiguousarray(boards)).cuda(), reward_fn=kind)
        return a["state"].cpu().numpy(), a["reward"].cpu().numpy(), a["valid_actions"].cpu().numpy().astype(bool)

    return move


def _guarded(shape, dtype, dev, pad: int = 64):
    """a tensor inside a buffer of canary words, and a check that the canaries are intact"""
    n = int(np.prod(shape))
    nbytes = n * torch.empty(0, dtype=dtype).element_size()
    buf = torch.full((2 * pad + (nbytes + 3) // 4,), CANARY, dtype=torch.int32, device=dev)
    clean = buf.clone().view(torch.uint8)
    raw = buf.view(torch.uint8)
    body = raw[4 * pad:4 * pad + nbytes].view(dtype).view(shape)

    def intact():
        assert torch.equal(raw[:4 * pad], clean[:4 * pad]), "bytes before the buffer were written"
        assert torch.equal(raw[4 * pad + nbytes:], clean[4 * pad + nbytes:]), "bytes after the buffer were written"

    return body, intact


def _guarded_out(m: int, action_dtype, dev):
    outs, checks = {}, []
    for key, shape, dtype in (("action", (m,), action_dtype), ("state", (m, 16), torch.uint8), ("reward", (m,), torch.float32),
                              ("value", (m,), torch.float32), ("q", (m, 4), torch.float32)):
        outs[key], ok = _guarded(shape, dtype, dev)
        checks.append(ok)
    return outs, lambda: [c() for c in checks]


def _same_bits(got: np.ndarray, want: np.ndarray, what: str) -> None:
    """bit-identical float32, except that a NaN matches any NaN (payloads differ between the device and NumPy)"""
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=what)
    np.testing.assert_array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32), err_msg=what)


def _check(got: dict, want: dict, rows=None) -> None:
    g = {k: v.cpu().numpy() for k, v in got.items()}
    if rows is not None:
        g = {k: v[rows] for k, v in g.items()}
    np.testing.assert_array_equal(g["action"].astype(np.int64), want["action"], err_msg="action")
    np.testing.assert_array_equal(g["state"], want["state"], err_msg="state")
    _same_bits(g["reward"], want["reward"], "reward")
    _same_bits(g["value"], want["value"], "value")
    _same_bits(g["q"], want["q"], "q")


def _run_and_check(ops, pool, w, tuples, kind, two_prob, depth, sizes):
    dev = _gpu()
    w_dev = torch.from_numpy(w).to(dev)
    want = xref.expectimax(pool, w, tuples, depth=depth, two_prob=two_prob, move=_move(ops, kind))
    for m in sizes:
        b = torch.from_numpy(pool[:m]).to(dev)
        for dtype in (torch.int64, torch.uint8):
            out, intact = _guarded_out(m, dtype, dev)
            got = ops.ntuple_expectimax(b, w_dev, tuples, depth=depth, two_prob=two_prob, reward_fn=kind, action_dtype=dtype, out=out)
            assert all(got[k].data_ptr() == out[k].data_ptr() for k in out)
            intact()
            _check(got, {k: v[:m] for k, v in want.items()})
    return want


# ---- depth 1 ----------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def played():
    return np.concatenate([_played_boards(256, 60, 1), _played_boards(256, 300, 2)])


@pytest.mark.gpu
@pytest.mark.parametrize("two_prob", TWO_PROBS)
@pytest.mark.parametrize("kind", KINDS)
def test_depth1_bit_exact(ops, played, kind, two_prob):
    rng = np.random.default_rng(KINDS.index(kind) * 10 + TWO_PROBS.index(two_prob))
    pool = _pool(rng, 300, played, 0.4)
    for shape in ("k1", "k4", "k16"):
        tuples = _tuples(rng, shape)
        for weights in ("random", "zero", "naninf"):
            _run_and_check(ops, pool, _weights(rng, tuples, weights), tuples, kind, two_prob, 1, (1, 255, 257, pool.shape[0]))


@pytest.mark.gpu
def test_depth1_large_batch_sampled_rows(ops, played):
    dev = _gpu()
    rng = np.random.default_rng(50)
    tuples = ref.STANDARD_4X6
    w = _weights(rng, tuples, "random")
    pool = _pool(rng, 4000, played, 0.4)
    m = (1 << 20) + 3
    idx = rng.integers(0, pool.shape[0], m)
    boards = pool[idx]
    got = ops.ntuple_expectimax(torch.from_numpy(boards).to(dev), torch.from_numpy(w).to(dev), tuples, two_prob=0.8, reward_fn="normal")
    rows = np.unique(np.concatenate([np.arange(2048), np.arange(m - 2048, m), rng.integers(0, m, 4096)]))
    want = xref.expectimax(boards[rows], w, tuples, depth=1, two_prob=0.8, move=_move(ops, "normal"))
    _check(got, want, rows)


# ---- depth 2 ----------------------------------------------------------------------------------------

DEPTH2_CASES = [("normal", 0.8, "random", "k4"), ("improved", 0.0, "zero", "k1"), ("rank", 1.0, "naninf", "k16"),
                ("maxcell", 0.3, "random", "k4")]


@pytest.mark.gpu
@pytest.mark.parametrize("case", DEPTH2_CASES, ids=lambda c: "-".join(map(str, c)))
def test_depth2_bit_exact(ops, played, case):
    kind, two_prob, weights, shape = case
    rng = np.random.default_rng(60 + DEPTH2_CASES.index(case))
    sub = played[rng.permutation(played.shape[0])[:40]]
    pool = _pool(rng, 260, sub, 0.3)
    tuples = _tuples(rng, shape)
    t0 = time.perf_counter()
    _run_and_check(ops, pool, _weights(rng, tuples, weights), tuples, kind, two_prob, 2, (1, 255, 257, pool.shape[0]))
    print(f"depth 2 {case}: {pool.shape[0]} boards, {time.perf_counter() - t0:.1f} s")


# ---- CUDA graphs, the network class, the policy -------------------------------------------------------


@pytest.mark.gpu
def test_graph_replay_equals_eager(ops, played):
    dev = _gpu()
    rng = np.random.default_rng(70)
    tuples = ref.STANDARD_4X6
    w = torch.from_numpy(_weights(rng, tuples, "random")).to(dev)
    m = 3001
    static_b = torch.zeros((m, 16), dtype=torch.uint8, device=dev)
    outs = {d: {"action": torch.empty((m,), dtype=torch.uint8, device=dev), "state": torch.empty((m, 16), dtype=torch.uint8, device=dev),
                "reward": torch.empty((m,), dtype=torch.float32, device=dev), "value": torch.empty((m,), dtype=torch.float32, device=dev),
                "q": torch.empty((m, 4), dtype=torch.float32, device=dev)} for d in (1, 2)}

    def run():
        for d in (1, 2):
            ops.ntuple_expectimax(static_b, w, tuples, depth=d, two_prob=0.9, reward_fn="rank", action_dtype=torch.uint8, out=outs[d])

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):  # warm-up outside the capture
        run()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run()
    for rep in range(3):
        pool = _pool(rng, m, played, 0.3 + 0.2 * rep)[:m]
        b = torch.from_numpy(pool).to(dev)
        static_b.copy_(b)
        graph.replay()
        for d in (1, 2):
            eager = ops.ntuple_expectimax(b, w, tuples, depth=d, two_prob=0.9, reward_fn="rank", action_dtype=torch.uint8)
            for k in eager:
                assert torch.equal(outs[d][k].view(torch.uint8), eager[k].view(torch.uint8)), (d, k)


@pytest.mark.gpu
def test_network_method_policy_and_runner(ops):
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import ExpectimaxPolicy, NTupleNetwork
    from ml2048_b200.runner import DeviceRunner

    dev = _gpu()
    net = NTupleNetwork(((0, 1, 2, 3), (4, 5, 6, 7), (0, 4, 8, 12)), device=dev)
    net.weights.copy_(torch.randn(net.weights.numel(), device=dev) * 100)
    env = VecGame(512, "improved", two_prob=0.7, output="torch", sync_free=True)
    env.reset(1)
    b = env.observations()[0]
    for d in (1, 2):
        got = net.expectimax(b, depth=d, two_prob=0.7, reward_fn="improved")
        want = ops.ntuple_expectimax(b, net.weights, net.tuples, depth=d, two_prob=0.7, reward_fn="improved")
        for k in want:
            assert torch.equal(got[k].view(torch.uint8), want[k].view(torch.uint8)), k
    # as a DeviceRunner policy it plays what ops.ntuple_expectimax chooses
    for depth in (1, 2):
        pol = ExpectimaxPolicy(net, depth=depth, reward_fn="improved", two_prob=0.7)
        runner = DeviceRunner(env, 512)
        seen = []
        runner.add_callback("prepared", lambda e, idx: seen.append(("board", e.observations()[0].clone())))
        runner.add_callback("stepped", lambda e, res, actions, lp: seen.append(("action", actions.clone(), lp.clone())))
        for _ in range(6):
            runner.step_once(pol)
        assert len(seen) == 12
        for (_, board), (_, actions, lp) in zip(seen[0::2], seen[1::2]):
            want = ops.ntuple_expectimax(board, net.weights, net.tuples, depth=depth, two_prob=0.7, reward_fn="improved")["action"]
            assert torch.equal(actions.to(dev), want) and not bool(lp.any())


# ---- strength ---------------------------------------------------------------------------------------


def _play_to_the_end(net, choose, games: int, seed: int, max_steps: int = 200000):
    """every game from reset to its end (episode log of ids < games); (score, length) per game, wall seconds per move"""
    from ml2048_b200 import VecGame

    env = VecGame(games, output="torch", sync_free=True, rng_mode="philox", track_merged=False)
    env.reset(seed)
    env.enable_episode_log(games)
    log = env.episode_log()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    steps = 0
    while steps < max_steps:
        env.prepare()
        env.step(choose(env.observations()[0]))
        steps += 1
        if steps % 64 == 0 and bool((log["max_tile"] > 0).all()):
            break
    torch.cuda.synchronize()
    assert bool((log["max_tile"] > 0).all()), "some game did not end"
    return log["score"].cpu().numpy().astype(np.float64), log["steps"].cpu().numpy(), (time.perf_counter() - t0) / steps


@pytest.mark.gpu
def test_expectimax_beats_greedy_on_trained_weights(ops):
    """Train the standard 4x6 network as test_learner_beats_the_random_policy does (M = 2^14, 100 000 steps), then play the
    same 2048 games (same Philox seed) from reset to their end with the greedy move and with depth-1 expectimax.

    Measured on one B200 at a 1000 W limit: greedy mean score 22 435 (mean length 1 148), depth-1 expectimax 39 270 (1 816),
    a gain of 16 835; the margin is about half of that gain."""
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner

    dev = _gpu()
    net = NTupleNetwork(device=dev)
    env = VecGame(1 << 14, output="torch", sync_free=True, rng_mode="philox")
    learner = TDAfterstateLearner(env, net)
    learner.reset(7)
    for _ in range(100000):
        learner.step()
    torch.cuda.synchronize()
    out = {"action": torch.empty((2048,), dtype=torch.uint8, device=dev), "state": torch.empty((2048, 16), dtype=torch.uint8, device=dev),
           "reward": torch.empty((2048,), dtype=torch.float32, device=dev), "value": torch.empty((2048,), dtype=torch.float32, device=dev),
           "q": torch.empty((2048, 4), dtype=torch.float32, device=dev)}
    greedy = _play_to_the_end(net, lambda b: net.greedy(b, action_dtype=torch.uint8)["action"], 2048, 11)
    expecti = _play_to_the_end(net, lambda b: net.expectimax(b, depth=1, action_dtype=torch.uint8, out=out)["action"], 2048, 11)
    g_mean, x_mean = greedy[0].mean(), expecti[0].mean()
    print(f"greedy: mean score {g_mean:.0f}, mean length {greedy[1].mean():.0f}, {greedy[2] * 1e6:.0f} us/move; "
          f"expectimax depth 1: mean score {x_mean:.0f}, mean length {expecti[1].mean():.0f}, {expecti[2] * 1e6:.0f} us/move")
    assert x_mean > g_mean + MARGIN, (g_mean, x_mean)


MARGIN = 8000.0
