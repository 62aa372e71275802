"""
N-tuple networks on the GPU (``ops.ntuple_value``, ``ops.ntuple_greedy``, ``ops.ntuple_td_update``, ``ml2048_b200.ntuple``)
against the NumPy definition in tests/_ntuple_ref.py.

- value: bit-exact, random non-zero weights, K = 1 / 4 / 16 with lengths 1..6, boards from a played environment plus boards
  with cells 15, 16, 17 and arbitrary bytes, M = 1, 255, 256, 257, 2^20 + 3, and M = 2^27 + 1 where board byte offsets pass
  2^31 (sampled rows); canary words around every output.
- greedy: bit-exact (action, afterstate, reward, value) against ``ops.afterstates`` + the reference's V and tie rule for all
  four reward kinds, zero weights (ties everywhere), dead boards, NaN and -inf weights, int64 and uint8 actions, and sampled
  rows against the C oracle's ``board_move`` / ``board_reward``.
- td_update: delta bit-exact against the pre-call weights; weights bit-exact for one game per call and for games with
  disjoint entries; many games on shared entries within n * 2^-24 * (|w0| + sum |delta|) of float64 (n = adds to that
  entry); masked-out games and untouched entries bitwise unchanged; canaries on both sides of the weights and of delta.
- CUDA graphs: value + greedy replayed equal eager bit for bit; td_update replayed within the tolerance above.
- Learning: TDAfterstateLearner from zero weights at M = 2^14 clearly beats the random policy (see the test's docstring).
"""

from __future__ import annotations

import time

import numpy as np
import pytest
import torch

import _ntuple_ref as ref
from _ntuple_gpu import _gpu, ops  # noqa: F401 (ops is a fixture)

KINDS = ("normal", "improved", "rank", "maxcell")
CANARY = 0x5A5A5A5A


def _boards(rng, m: int) -> np.ndarray:
    """a mixture: 40 % empty cells with exponents 1..15, full boards (dead ones among them), small exponents (ties), cells
    15 / 16 / 17, and arbitrary bytes"""
    u = rng.random((m, 16))
    b = np.where(u < 0.4, 0, rng.integers(1, 16, size=(m, 16))).astype(np.uint8)
    k = max(m // 8, 1)
    b[k:2 * k] = rng.integers(1, 16, size=b[k:2 * k].shape)
    b[2 * k:3 * k] = rng.integers(0, 3, size=b[2 * k:3 * k].shape)
    b[3 * k:4 * k] = rng.choice(np.array([0, 14, 15, 16, 17], np.uint8), size=b[3 * k:4 * k].shape)
    b[4 * k:5 * k] = rng.integers(0, 256, size=b[4 * k:5 * k].shape, dtype=np.uint8)
    return b


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


def _tuples(rng, k: int, lengths=None):
    lengths = lengths if lengths is not None else rng.integers(1, 7, size=k)
    return tuple(tuple(int(c) for c in rng.permutation(16)[:n]) for n in lengths)


def _weights(rng, tuples, scale=100.0) -> np.ndarray:
    w = (rng.standard_normal(ref.num_weights(tuples)) * scale).astype(np.float32)
    w[w == 0] = 1.0
    return w


def _guarded(n: int, dtype, dev, fill=None, pad: int = 64):
    """a (n,) tensor inside a buffer of canary words, and a check that the canaries are intact"""
    nbytes = n * torch.empty(0, dtype=dtype).element_size()
    buf = torch.full((2 * pad + (nbytes + 3) // 4,), CANARY, dtype=torch.int32, device=dev)
    clean = buf.clone().view(torch.uint8)
    raw = buf.view(torch.uint8)
    body = raw[4 * pad:4 * pad + nbytes].view(dtype)
    if fill is not None:
        body.copy_(fill)

    def intact():
        assert torch.equal(raw[:4 * pad], clean[:4 * pad]), "bytes before the buffer were written"
        assert torch.equal(raw[4 * pad + nbytes:], clean[4 * pad + nbytes:]), "bytes after the buffer were written"

    return body, intact


# ---- value ----------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["k1", "k4", "k16"])
def test_value_bit_exact(ops, shape):
    rng = np.random.default_rng({"k1": 1, "k4": 2, "k16": 3}[shape])
    tuples = {"k1": ((3, 7, 11, 15, 14, 13),), "k4": ref.STANDARD_4X6, "k16": _tuples(rng, 16, [1, 2, 3, 4, 5, 6, 2, 3, 4, 5, 1, 2, 3, 4, 5, 6])}[shape]
    w = _weights(rng, tuples)
    dev = _gpu()
    w_dev, w_ok = _guarded(w.size, torch.float32, dev, torch.from_numpy(w))
    pool = np.concatenate([_played_boards(4096), _boards(rng, 8192)])
    for m in (1, 255, 256, 257, (1 << 20) + 3):
        boards = pool[rng.integers(0, pool.shape[0], m)] if m > pool.shape[0] else pool[:m]
        out, ok = _guarded(m, torch.float32, dev)
        got = ops.ntuple_value(torch.from_numpy(boards).to(dev), w_dev, tuples, out=out)
        assert got.data_ptr() == out.data_ptr()
        ok()
        np.testing.assert_array_equal(got.cpu().numpy().view(np.uint32), ref.value(boards, w, tuples).view(np.uint32))
    w_ok()
    assert torch.equal(w_dev.cpu(), torch.from_numpy(w))
    # int8 boards read the same bytes
    b8 = torch.from_numpy(pool[:1000]).to(dev)
    assert torch.equal(ops.ntuple_value(b8.view(torch.int8), w_dev, tuples), ops.ntuple_value(b8, w_dev, tuples))


@pytest.mark.gpu
def test_value_beyond_2gib_of_boards(ops):
    """M = 2^27 + 1: board byte offsets pass 2^31.  Rows at both ends and a seeded sample against the reference."""
    dev = _gpu()
    rng = np.random.default_rng(4)
    tuples = ref.STANDARD_4X6
    w = _weights(rng, tuples)
    m = (1 << 27) + 1
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    boards = torch.randint(0, 18, (m, 16), dtype=torch.uint8, device=dev, generator=g)
    got = ops.ntuple_value(boards, torch.from_numpy(w).to(dev), tuples)
    rows = np.unique(np.concatenate([np.arange(4096), np.arange(m - 4096, m), rng.integers(0, m, 65536)]))
    idx = torch.from_numpy(rows).to(dev)
    b = boards[idx].cpu().numpy()
    np.testing.assert_array_equal(got[idx].cpu().numpy().view(np.uint32), ref.value(b, w, tuples).view(np.uint32))
    del boards, got
    torch.cuda.empty_cache()


# ---- greedy ---------------------------------------------------------------------------------------


def _greedy_ref(ops, boards_dev, w, tuples, kind):
    a = ops.afterstates(boards_dev, reward_fn=kind)
    return ref.greedy(boards_dev.cpu().numpy(), a["state"].cpu().numpy(), a["reward"].cpu().numpy(),
                      a["valid_actions"].cpu().numpy(), w, tuples)


def _same_bits(got: np.ndarray, want: np.ndarray) -> None:
    """bit-identical float32, except that a NaN matches any NaN (the device's NaN payload is 0x7fffffff, NumPy's 0x7fc00000)"""
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan)
    np.testing.assert_array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))


def _check_greedy(got: dict, want: dict) -> None:
    np.testing.assert_array_equal(got["action"].cpu().numpy().astype(np.int64), want["action"])
    np.testing.assert_array_equal(got["state"].cpu().numpy(), want["state"])
    np.testing.assert_array_equal(got["reward"].cpu().numpy().view(np.uint32), want["reward"].view(np.uint32))
    _same_bits(got["value"].cpu().numpy(), want["value"])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_greedy_bit_exact(ops, oracle, kind):
    dev = _gpu()
    rng = np.random.default_rng(KINDS.index(kind) + 10)
    pool = np.concatenate([_played_boards(8192), _boards(rng, 20000)])
    pool[1::53] = pool[0::53][:pool[1::53].shape[0]]  # repeated boards
    dead = np.tile(np.array([1, 2, 1, 2, 2, 1, 2, 1], np.uint8), 2)  # a checkerboard: no valid move
    pool[::97] = dead
    for tuples in (ref.STANDARD_4X6, _tuples(rng, 5)):
        for weights in ("random", "zero", "small"):
            w = {"random": _weights(rng, tuples, 1000.0), "zero": np.zeros(ref.num_weights(tuples), np.float32),
                 "small": rng.integers(-2, 3, ref.num_weights(tuples)).astype(np.float32)}[weights]
            w_dev = torch.from_numpy(w).to(dev)
            for m in (1, 257, pool.shape[0]):
                b = torch.from_numpy(pool[:m]).to(dev)
                want = _greedy_ref(ops, b, w, tuples, kind)
                for dtype in (torch.int64, torch.uint8):
                    got = ops.ntuple_greedy(b, w_dev, tuples, reward_fn=kind, action_dtype=dtype)
                    assert got["action"].dtype == dtype
                    _check_greedy(got, want)
    # sampled rows against the C oracle's move and reward
    got = {k: v.cpu().numpy() for k, v in ops.ntuple_greedy(torch.from_numpy(pool).to(dev), w_dev, tuples, reward_fn=kind).items()}
    for i in rng.integers(0, pool.shape[0], 400):
        bd = pool[i]
        if bd.max() > 15:
            continue  # the oracle logs fusions of exponents below 16 only
        a = int(got["action"][i])
        nb, mg = oracle.board_move(bd, a)
        np.testing.assert_array_equal(got["state"][i], nb)
        moved = bool((nb != bd).any())
        assert got["reward"][i] == (oracle.board_reward(kind, nb, bd, mg) if moved else 0.0)
    assert (got["action"][::97] == 0).all() and (got["state"][::97] == dead).all()
    assert (got["reward"][::97] == 0).all() and (got["value"][::97] == 0).all()


@pytest.mark.gpu
def test_greedy_nan_and_inf_weights(ops):
    """NaN q ranks as -inf: a number beats it, and where every valid q is NaN or -inf the smallest valid direction wins"""
    dev = _gpu()
    rng = np.random.default_rng(20)
    tuples = ((0, 1, 2, 3), (4, 5, 6, 7), (0, 4, 8, 12))
    pool = _boards(rng, 50000)
    b = torch.from_numpy(pool).to(dev)
    n = ref.num_weights(tuples)
    after = ops.afterstates(b)
    valid = after["valid_actions"].cpu().numpy().astype(bool)
    first_valid = np.where(valid.any(axis=1), valid.argmax(axis=1), 0)
    for w in (np.full(n, np.nan, np.float32), np.full(n, -np.inf, np.float32)):
        got = ops.ntuple_greedy(b, torch.from_numpy(w).to(dev), tuples)
        np.testing.assert_array_equal(got["action"].cpu().numpy(), first_valid)
        _check_greedy(got, _greedy_ref(ops, b, w, tuples, "normal"))
    for share in (0.01, 0.3, 0.9):
        w = _weights(rng, tuples)
        w[rng.random(n) < share] = np.nan
        w[rng.random(n) < share / 4] = -np.inf
        w[rng.random(n) < share / 8] = np.inf  # inf + -inf = NaN as well
        got = ops.ntuple_greedy(b, torch.from_numpy(w).to(dev), tuples, reward_fn="improved")
        _check_greedy(got, _greedy_ref(ops, b, w, tuples, "improved"))


# ---- TD(0) update -------------------------------------------------------------------------------------


def _disjoint_rows(boards, tuples, want: int) -> np.ndarray:
    """indices of boards whose entry sets are pairwise disjoint (and without repeats inside one board)"""
    used, keep = set(), []
    for i, row in enumerate(ref.entries(boards, tuples)):
        s = set(int(x) for x in row)
        if len(s) == row.size and not (s & used):
            used |= s
            keep.append(i)
            if len(keep) == want:
                break
    return np.array(keep, np.int64)


@pytest.mark.gpu
def test_td_update_exact_cases(ops):
    dev = _gpu()
    rng = np.random.default_rng(30)
    tuples = ((0, 1, 2, 3, 4, 5), (5, 6, 9, 10, 13), (3, 7, 11, 15, 14))
    n = ref.num_weights(tuples)
    w0 = _weights(rng, tuples)
    boards = _boards(rng, 20000)
    w_dev, w_ok = _guarded(n, torch.float32, dev, torch.from_numpy(w0))
    # one game per call (its own 8K adds may share entries: one thread adds them in order)
    w = w0.copy()
    for i in range(40):
        b = boards[i:i + 1]
        y = rng.standard_normal(1).astype(np.float32) * 50
        d_dev, d_ok = _guarded(1, torch.float32, dev)
        d = ops.ntuple_td_update(torch.from_numpy(b).to(dev), torch.from_numpy(y).to(dev), w_dev, tuples, alpha=0.0625,
                                 delta_out=d_dev)
        want_d = ref.td_delta(b, y, w, tuples, 0.0625)
        np.testing.assert_array_equal(d.cpu().numpy().view(np.uint32), want_d.view(np.uint32))
        w = ref.td_apply_f32(b, want_d, w, tuples)
        d_ok()
    np.testing.assert_array_equal(w_dev.cpu().numpy().view(np.uint32), w.view(np.uint32))
    # games whose entries are disjoint, with a mask
    uniform = rng.integers(0, 16, size=(20000, 16)).astype(np.uint8)  # few shared entries
    rows = _disjoint_rows(uniform, tuples, 2000)
    assert rows.size >= 500, rows.size
    b = uniform[rows]
    m = b.shape[0]
    y = (rng.standard_normal(m) * 100).astype(np.float32)
    mask = (rng.random(m) < 0.7).astype(np.uint8)
    for mask_dtype in (torch.uint8, torch.bool):
        before = w_dev.cpu().numpy().copy()
        d = ops.ntuple_td_update(torch.from_numpy(b).to(dev), torch.from_numpy(y).to(dev), w_dev, tuples, alpha=0.01,
                                 mask=torch.from_numpy(mask).to(dev, mask_dtype))
        want_d = ref.td_delta(b, y, before, tuples, 0.01, mask)
        np.testing.assert_array_equal(d.cpu().numpy().view(np.uint32), want_d.view(np.uint32))
        assert (d.cpu().numpy()[mask == 0] == 0).all()
        want_w = ref.td_apply_f32(b, want_d, before, tuples, mask)
        np.testing.assert_array_equal(w_dev.cpu().numpy().view(np.uint32), want_w.view(np.uint32))
    w_ok()


def _td_tolerance_check(got: np.ndarray, w0: np.ndarray, w64: np.ndarray, adds: np.ndarray, sabs: np.ndarray) -> None:
    touched = adds > 0
    np.testing.assert_array_equal(got[~touched].view(np.uint32), w0[~touched].view(np.uint32))
    err = np.abs(got[touched].astype(np.float64) - w64[touched])
    bound = adds[touched] * 2.0 ** -24 * (np.abs(w0[touched].astype(np.float64)) + sabs[touched])
    assert (err <= bound).all(), (err - bound).max()


@pytest.mark.gpu
@pytest.mark.parametrize("m", [4096, 1 << 18])
def test_td_update_colliding_games(ops, m):
    """early-game boards (few tiles, small exponents): thousands of adds land on the same entries"""
    dev = _gpu()
    rng = np.random.default_rng(31)
    tuples = ref.STANDARD_4X6
    n = ref.num_weights(tuples)
    w0 = _weights(rng, tuples, 10.0)
    b = np.where(rng.random((m, 16)) < 0.7, 0, rng.integers(1, 4, size=(m, 16))).astype(np.uint8)
    y = (rng.standard_normal(m) * 30).astype(np.float32)
    mask = (rng.random(m) < 0.8).astype(np.uint8)
    w_dev, w_ok = _guarded(n, torch.float32, dev, torch.from_numpy(w0))
    d_dev, d_ok = _guarded(m, torch.float32, dev)
    d = ops.ntuple_td_update(torch.from_numpy(b).to(dev), torch.from_numpy(y).to(dev), w_dev, tuples, alpha=0.003,
                             mask=torch.from_numpy(mask).to(dev), delta_out=d_dev)
    want_d = ref.td_delta(b, y, w0, tuples, 0.003, mask)
    np.testing.assert_array_equal(d.cpu().numpy().view(np.uint32), want_d.view(np.uint32))
    w64, adds, sabs = ref.td_apply_f64(b, want_d, w0, tuples, mask)
    assert adds.max() > 1000
    _td_tolerance_check(w_dev.cpu().numpy(), w0, w64, adds, sabs)
    w_ok()
    d_ok()


# ---- CUDA graphs ----------------------------------------------------------------------------------


@pytest.mark.gpu
def test_graph_replay_equals_eager(ops):
    dev = _gpu()
    rng = np.random.default_rng(40)
    tuples = ref.STANDARD_4X6
    n = ref.num_weights(tuples)
    w0 = _weights(rng, tuples, 10.0)
    m = 70001
    w = torch.from_numpy(w0).to(dev)
    static_b = torch.zeros((m, 16), dtype=torch.uint8, device=dev)
    static_y = torch.zeros((m,), dtype=torch.float32, device=dev)
    v_out = torch.empty((m,), dtype=torch.float32, device=dev)
    g_out = {"action": torch.empty((m,), dtype=torch.uint8, device=dev), "state": torch.empty((m, 16), dtype=torch.uint8, device=dev),
             "reward": torch.empty((m,), dtype=torch.float32, device=dev), "value": torch.empty((m,), dtype=torch.float32, device=dev)}
    d_out = torch.empty((m,), dtype=torch.float32, device=dev)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):  # warm-up outside the capture
        ops.ntuple_value(static_b, w, tuples, out=v_out)
        ops.ntuple_greedy(static_b, w, tuples, reward_fn="rank", action_dtype=torch.uint8, out=g_out)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ops.ntuple_value(static_b, w, tuples, out=v_out)
        ops.ntuple_greedy(static_b, w, tuples, reward_fn="rank", action_dtype=torch.uint8, out=g_out)
    td_graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(td_graph):
        ops.ntuple_td_update(static_b, static_y, w, tuples, alpha=0.002, delta_out=d_out)
    for rep in range(3):
        b = torch.from_numpy(_boards(rng, m)).to(dev)
        static_b.copy_(b)
        graph.replay()
        assert torch.equal(v_out.view(torch.int32), ops.ntuple_value(b, w, tuples).view(torch.int32))
        eager = ops.ntuple_greedy(b, w, tuples, reward_fn="rank", action_dtype=torch.uint8)
        for k in g_out:
            assert torch.equal(g_out[k].view(torch.uint8), eager[k].view(torch.uint8)), k
        # td_update: replay on one copy of the weights, eager on another, both from the same start
        start = w.clone()
        y = torch.randn(m, device=dev) * 20
        static_y.copy_(y)
        td_graph.replay()
        replayed = w.clone()
        w_eager = start.clone()
        d = ops.ntuple_td_update(b, y, w_eager, tuples, alpha=0.002)
        assert torch.equal(d_out.view(torch.int32), d.view(torch.int32))
        bh, dh = b.cpu().numpy(), d.cpu().numpy()
        w64, adds, sabs = ref.td_apply_f64(bh, dh, start.cpu().numpy(), tuples)
        _td_tolerance_check(replayed.cpu().numpy(), start.cpu().numpy(), w64, adds, sabs)
        _td_tolerance_check(w_eager.cpu().numpy(), start.cpu().numpy(), w64, adds, sabs)
    assert n == w.numel()


# ---- the network class and the learner -------------------------------------------------------------


@pytest.mark.gpu
def test_network_state_dict_and_policy(ops):
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import GreedyPolicy, NTupleNetwork, TDAfterstateLearner
    from ml2048_b200.runner import DeviceRunner

    dev = _gpu()
    net = NTupleNetwork(((0, 1, 2), (4, 5)), device=dev)
    assert net.weights.numel() == 16 ** 3 + 16 ** 2 and not bool(net.weights.any())
    assert net.offsets == [0, 4096]
    net.weights.copy_(torch.randn(net.weights.numel(), device=dev))
    other = NTupleNetwork(((0, 1, 2), (4, 5)), device=dev)
    other.load_state_dict(net.state_dict())
    assert torch.equal(other.weights, net.weights)
    with pytest.raises(ValueError):
        NTupleNetwork(((0, 1, 2), (4, 6)), device=dev).load_state_dict(net.state_dict())
    with pytest.raises(ValueError):
        TDAfterstateLearner(VecGame(64, output="torch"), net)
    # as a DeviceRunner policy it plays what greedy chooses
    env = VecGame(512, output="torch", sync_free=True)
    env.reset(1)
    runner = DeviceRunner(env, 512)
    seen = []
    runner.add_callback("stepped", lambda e, res, actions, lp: seen.append(actions.clone()))
    pol = GreedyPolicy(net)
    for _ in range(5):
        env.prepare()
        want = net.greedy(env.observations()[0])["action"].clone()
        board, valid = env.observations()
        got, lp = pol.sample_actions(board.long(), valid.bool())
        assert torch.equal(got, want) and not bool(lp.any())
        env.step(got)
    runner.step_once(pol)
    assert len(seen) == 1
    # alpha = 0: evaluation, the weights stay as they are
    w = net.weights.clone()
    env2 = VecGame(512, output="torch", sync_free=True)
    learner = TDAfterstateLearner(env2, net, alpha=0.0)
    learner.reset(2)
    for _ in range(20):
        learner.step()
    assert torch.equal(net.weights, w)


@pytest.mark.gpu
def test_learner_first_step_masks_and_terminal_targets(ops):
    """the first step after reset() updates nothing; a game that ended is updated toward 0"""
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner

    dev = _gpu()
    net = NTupleNetwork(device=dev)
    env = VecGame(4096, output="torch", sync_free=True)
    learner = TDAfterstateLearner(env, net, alpha=0.01)
    learner.reset(3)
    learner.step()
    assert not bool(net.weights.any()) and not bool(learner.delta.any())
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


@pytest.mark.gpu
def test_learner_beats_the_random_policy(ops):
    """TD(0) afterstate learning from zero weights, M = 2^14 games, the standard 4x6 network, the default alpha, a fixed
    number of steps (100 000 steps, 8.7 s on one B200 at 1000 W).  The random policy (tests/golden/random_policy_stats.npz, 16
    seeds of the live reference): mean score 1 015, mean length 106 steps, 512 reached in 0.014 % of episodes.

    Measured on that B200 over the 380 805 episodes that end in the last quarter of the run: mean score 20 668, 512 reached in
    98.4 %, 1024 in 84.6 %, 2048 in 35.0 %.  The thresholds are about half of the score and of the 512 share."""
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner

    dev = _gpu()
    net = NTupleNetwork(device=dev)
    env = VecGame(1 << 14, output="torch", sync_free=True, rng_mode="philox")
    learner = TDAfterstateLearner(env, net)
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
    print(f"learner: {steps} steps in {elapsed:.1f} s, {eps} episodes in the last quarter, mean score {mean_score:.0f}, "
          f">= 512: {share512:.3f}, >= 1024: {hist[10:].sum() / max(eps, 1):.3f}, >= 2048: {hist[11:].sum() / max(eps, 1):.4f}")
    assert eps > 100
    assert mean_score > THRESHOLDS["mean_score"], mean_score
    assert share512 > THRESHOLDS["share512"], share512


LEARN_STEPS = 100000
THRESHOLDS = {"mean_score": 10000.0, "share512": 0.5}
