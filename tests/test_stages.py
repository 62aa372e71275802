"""
Multi-stage n-tuple networks on the GPU (the ``stages=`` argument of ``ops.ntuple_*``, ``NTupleNetwork(stages=...)``) against
the NumPy definition in tests/_stage_ref.py.

- S = 2, 3 and 8 (stages (4,), (4, 6) and (2, ..., 8)), each stage with its own seeded weights.  Boards: played games,
  boards whose largest tile is exactly tau - 1, tau and tau + 1 for every threshold, boards with cells >= 16, and for
  expectimax boards whose moves (a merge into tau) or spawns (a 4 onto a board of 2s) cross a threshold inside the search.
- Bit for bit: value; greedy with uint8 and int64 actions; expectimax at depth 1 and 2 for every reward kind and two_prob
  0.9 / 1 / 0; the delta of TD(0), TC, TD(lambda) and TC(lambda).  The weights, coherence and accumulator too, on data whose
  every sum is exact in float32 (integer weights and targets, alpha = 1/16, lambda = 1/2), so that the order of the atomics
  cannot change a bit.  Canary words around every S * N buffer; the entries of every stage that no masked-in x_0 is in stay
  bit for bit.
- S = 1: ``stages=()`` and an explicit S = 1 call of each ``ml2048_staged_*`` entry equal the single-stage entry bit for bit.
- CUDA-graph replay of a staged learner step (greedy, then TD(0), TC or TD(lambda) with h = 3) equals the eager step.
- ``TDAfterstateLearner`` on a staged network, ``GreedyPolicy`` and ``ExpectimaxPolicy`` under ``DeviceRunner``.
"""

from __future__ import annotations

import numpy as np
import pytest
import torch

import _lambda_ref as lref
import _ntuple_ref as nref
import _stage_ref as sref
from _ntuple_gpu import _gpu, ops  # noqa: F401 (ops is a fixture)

CANARY = 0x5A5A5A5A
KINDS = ("normal", "improved", "rank", "maxcell")
SMALL = ((0, 1, 2, 3), (4, 5, 6, 7), (0, 4, 8, 12), (1, 5, 9, 13))
CASES = {"s2": ((4,), nref.STANDARD_4X6), "s3": ((4, 6), SMALL), "s8": (tuple(range(2, 9)), SMALL)}


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


def _same_bits(got: np.ndarray, want: np.ndarray, what: str = "") -> None:
    """bit-identical float32, except that a NaN matches any NaN"""
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=what)
    np.testing.assert_array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32), err_msg=what)


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


def _edge_boards(rng, stages, per: int = 12, top: int = 17) -> np.ndarray:
    """largest tile exactly tau - 1, tau and tau + 1 for every threshold, random lower tiles and empty cells; then boards
    with cells 16..top"""
    out = []
    for tau in stages:
        for m in (tau - 1, tau, tau + 1):
            if not 0 <= m <= 15:
                continue
            b = np.where(rng.random((per, 16)) < 0.4, 0, rng.integers(1, max(m, 1) + 1, size=(per, 16))).astype(np.uint8)
            b = np.minimum(b, m)
            b[np.arange(per), rng.integers(0, 16, size=per)] = m
            out.append(b)
    hi = np.where(rng.random((per, 16)) < 0.4, 0, rng.integers(1, top + 1, size=(per, 16))).astype(np.uint8)
    hi[:, 5] = rng.integers(16, top + 1, size=per)
    out.append(hi)
    return np.concatenate(out)


def _crossing_boards(stages) -> np.ndarray:
    """boards whose moves or spawns cross a threshold inside the search: two adjacent tau - 1 tiles (a merge makes tau), and
    a board of 2s and one 4-spawn away from tau = 2"""
    out = []
    for tau in stages:
        if tau < 2:
            continue
        b = np.zeros(16, np.uint8)
        b[0] = b[1] = tau - 1
        b[6] = max(tau - 2, 1)
        out.append(b)
        c = b.copy()
        c[[0, 4]] = tau - 1, tau - 1  # vertical pair
        c[1] = 0
        out.append(c)
    two = np.zeros(16, np.uint8)
    two[[0, 5, 10]] = 1
    out.append(two)
    return np.stack(out)


def _stage_weights(rng, tuples, stages, scale=100.0, integer=False) -> np.ndarray:
    """distinct seeded weights per stage"""
    n = nref.num_weights(tuples)
    parts = []
    for s in range(len(stages) + 1):
        r = np.random.default_rng(rng.integers(1 << 30) + s)
        parts.append(r.integers(-8, 9, size=n).astype(np.float32) if integer else (r.standard_normal(n) * scale).astype(np.float32))
    return np.concatenate(parts)


@pytest.fixture(scope="module")
def played():
    return np.concatenate([_played_boards(512, 40, 1), _played_boards(512, 150, 2), _played_boards(512, 400, 3)])


def _afterstate_move(ops, kind):
    def move(boards: np.ndarray):
        a = ops.afterstates(torch.from_numpy(np.ascontiguousarray(boards)).cuda(), reward_fn=kind)
        return a["state"].cpu().numpy(), a["reward"].cpu().numpy(), a["valid_actions"].cpu().numpy().astype(bool)

    return move


# ---- value, greedy, expectimax --------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_value_and_greedy_bit_exact(ops, played, case):
    dev = _gpu()
    stages, tuples = CASES[case]
    rng = np.random.default_rng(list(CASES).index(case))
    w = _stage_weights(rng, tuples, stages)
    boards = np.concatenate([played, _edge_boards(rng, stages), _crossing_boards(stages)])
    st = sref.stage(boards, stages)
    assert set(st.tolist()) == set(range(len(stages) + 1)), "some stage has no board"
    w_dev, w_ok = _guarded((w.size,), torch.float32, dev, torch.from_numpy(w))
    b = torch.from_numpy(boards).to(dev)
    # value, also on arbitrary bytes
    anyb = np.concatenate([boards, rng.integers(0, 256, size=(300, 16), dtype=np.uint8)])
    got = ops.ntuple_value(torch.from_numpy(anyb).to(dev), w_dev, tuples, stages=stages).cpu().numpy()
    _same_bits(got, sref.value(anyb, w, tuples, stages), "value")
    # greedy, every reward kind, both action dtypes
    for kind in KINDS:
        after, reward, valid = _afterstate_move(ops, kind)(boards)
        want = sref.greedy(boards, after, reward, valid, w, tuples, stages)
        for dtype in (torch.uint8, torch.int64):
            g = ops.ntuple_greedy(b, w_dev, tuples, reward_fn=kind, action_dtype=dtype, stages=stages)
            assert g["action"].dtype == dtype
            np.testing.assert_array_equal(g["action"].cpu().numpy().astype(np.int64), want["action"])
            np.testing.assert_array_equal(g["state"].cpu().numpy(), want["state"])
            _same_bits(g["reward"].cpu().numpy(), want["reward"], "reward")
            _same_bits(g["value"].cpu().numpy(), want["value"], "value")
    w_ok()
    assert torch.equal(w_dev.cpu(), torch.from_numpy(w))


@pytest.mark.gpu
@pytest.mark.parametrize("depth", [1, 2])
@pytest.mark.parametrize("case", list(CASES))
def test_expectimax_bit_exact(ops, played, case, depth):
    dev = _gpu()
    stages, tuples = CASES[case]
    rng = np.random.default_rng(10 + list(CASES).index(case))
    w = _stage_weights(rng, tuples, stages)
    pool = np.concatenate([_crossing_boards(stages), _edge_boards(rng, stages, per=2 if depth == 2 else 8, top=17),
                           played[rng.permutation(played.shape[0])[:24 if depth == 2 else 400]]])
    w_dev = torch.from_numpy(w).to(dev)
    b = torch.from_numpy(pool).to(dev)
    for kind in KINDS:
        for two_prob in (0.9, 1.0, 0.0):
            want = sref.expectimax(pool, w, tuples, stages, depth=depth, two_prob=two_prob, move=_afterstate_move(ops, kind))
            dtype = torch.uint8 if two_prob == 0.9 else torch.int64
            got = ops.ntuple_expectimax(b, w_dev, tuples, depth=depth, two_prob=two_prob, reward_fn=kind, action_dtype=dtype,
                                        stages=stages)
            g = {k: v.cpu().numpy() for k, v in got.items()}
            what = f"{kind} two_prob={two_prob}"
            np.testing.assert_array_equal(g["action"].astype(np.int64), want["action"], err_msg=what)
            np.testing.assert_array_equal(g["state"], want["state"], err_msg=what)
            for k in ("reward", "value", "q"):
                _same_bits(g[k], want[k], f"{k} {what}")


# ---- updates ----------------------------------------------------------------------------------------------


def _exact_update_data(rng, boards, tuples, stages):
    """integer weights and targets, a mask: with alpha = 1/16 every delta and every sum of them is exact in float32"""
    w = _stage_weights(rng, tuples, stages, integer=True)
    m = boards.shape[0]
    target = rng.integers(-64, 65, size=m).astype(np.float32)
    mask = (rng.random(m) < 0.8).astype(np.uint8)
    coh = (rng.integers(-20, 21, size=(w.size, 2))).astype(np.float32)
    coh[:, 1] = np.abs(coh[:, 1]) + np.abs(coh[:, 0])
    coh[::3] = 0.0
    return w, target, mask, coh


def _untouched(before: np.ndarray, after: np.ndarray, x0: np.ndarray, mask, tuples, stages):
    """every entry of a stage that no masked-in x_0 is in stays bit for bit"""
    n = nref.num_weights(tuples)
    hit = set(sref.stage(x0[np.asarray(mask).astype(bool)], stages).tolist())
    for s in range(len(stages) + 1):
        if s not in hit:
            np.testing.assert_array_equal(after[s * n:(s + 1) * n].view(np.uint32), before[s * n:(s + 1) * n].view(np.uint32))
    return hit


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc"])
@pytest.mark.parametrize("case", list(CASES))
def test_target_updates_exact(ops, played, case, rule):
    dev = _gpu()
    stages, tuples = CASES[case]
    rng = np.random.default_rng(20 + list(CASES).index(case))
    boards = np.concatenate([played, _edge_boards(rng, stages)])
    alpha = 0.0625
    for subset in ("all", "low"):
        x0 = boards if subset == "all" else boards[sref.stage(boards, stages) < len(stages)]  # the top stage untouched
        w, target, mask, coh = _exact_update_data(rng, x0, tuples, stages)
        n = w.size
        w_dev, w_ok = _guarded((n,), torch.float32, dev, torch.from_numpy(w))
        d_dev, d_ok = _guarded((x0.shape[0],), torch.float32, dev)
        a = torch.from_numpy(x0).to(dev)
        t = torch.from_numpy(target).to(dev)
        mk = torch.from_numpy(mask).to(dev)
        want_d = sref.td_delta(x0, target, w, tuples, stages, alpha, mask)
        if rule == "td0":
            ops.ntuple_td_update(a, t, w_dev, tuples, alpha=alpha, mask=mk, delta_out=d_dev, stages=stages)
            want_w = sref.td_apply_f32(x0, want_d, w, tuples, stages, mask)
        else:
            c_dev, c_ok = _guarded((n, 2), torch.float32, dev, torch.from_numpy(coh))
            acc, acc_ok = _guarded((n, 2), torch.float32, dev, torch.zeros((n, 2)))
            ops.ntuple_tc_update(a, t, w_dev, c_dev, acc, tuples, alpha=alpha, mask=mk, delta_out=d_dev, stages=stages)
            want_w, want_c = sref.tc_update_f32(x0, want_d, w, coh, tuples, stages, mask)
            _same_bits(c_dev.cpu().numpy(), want_c, "coherence")
            assert not bool(acc.view(torch.int32).any()), "the accumulator is not all zero bits"
            c_ok(), acc_ok()
        _same_bits(d_dev.cpu().numpy(), want_d, "delta")
        got_w = w_dev.cpu().numpy()
        _same_bits(got_w, want_w, "weights")
        hit = _untouched(w, got_w, x0, mask, tuples, stages)
        assert (subset == "low") == (len(stages) not in hit)
        w_ok(), d_ok()


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc"])
@pytest.mark.parametrize("case", list(CASES))
def test_lambda_updates_exact(ops, played, case, rule):
    dev = _gpu()
    stages, tuples = CASES[case]
    rng = np.random.default_rng(30 + list(CASES).index(case))
    pool = np.concatenate([played, _edge_boards(rng, stages)])
    h, newest, lam, alpha = 3, 1, 0.5, 0.0625
    m = 1500
    ring = pool[rng.integers(0, pool.shape[0], size=(h + 1, m))]
    reward = rng.choice(np.array([0, 4, 8, 16, 256], np.float32), size=(h + 1, m))
    ended = (rng.random((h + 1, m)) < 0.1).astype(np.uint8)
    w, _, mask, coh = _exact_update_data(rng, ring[0], tuples, stages)
    n = w.size
    w_dev, w_ok = _guarded((n,), torch.float32, dev, torch.from_numpy(w))
    d_dev = torch.empty(m, device=dev)
    args = (torch.from_numpy(ring).to(dev), torch.from_numpy(reward).to(dev), torch.from_numpy(ended).to(dev), newest)
    mk = torch.from_numpy(mask).to(dev)
    want_d, x0 = sref.ring_delta(ring, reward, ended, newest, w, tuples, stages, lam, alpha, mask)
    if rule == "td0":
        ops.ntuple_td_lambda_update(*args, w_dev, tuples, alpha=alpha, lam=lam, mask=mk, delta_out=d_dev, stages=stages)
        want_w = sref.td_apply_f32(x0, want_d, w, tuples, stages, mask)
    else:
        c_dev, c_ok = _guarded((n, 2), torch.float32, dev, torch.from_numpy(coh))
        acc, acc_ok = _guarded((n, 2), torch.float32, dev, torch.zeros((n, 2)))
        ops.ntuple_tc_lambda_update(*args, w_dev, c_dev, acc, tuples, alpha=alpha, lam=lam, mask=mk, delta_out=d_dev, stages=stages)
        want_w, want_c = sref.tc_update_f32(x0, want_d, w, coh, tuples, stages, mask)
        _same_bits(c_dev.cpu().numpy(), want_c, "coherence")
        assert not bool(acc.view(torch.int32).any())
        c_ok(), acc_ok()
    _same_bits(d_dev.cpu().numpy(), want_d, "delta")
    _same_bits(w_dev.cpu().numpy(), want_w, "weights")
    _untouched(w, w_dev.cpu().numpy(), x0, mask, tuples, stages)
    w_ok()
    # the window boards are valued on their own stages: some window has boards of different stages
    win = lref.window(ring, newest)
    assert (sref.stage(win.reshape(-1, 16), stages).reshape(h + 1, m) != sref.stage(win[0], stages)[None]).any()


# ---- argument checks ------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_argument_errors(ops):
    """on CUDA tensors that are otherwise valid, so that the stage checks are the ones that fire: weights of N or 3N entries
    under two stages, coherence and accum of (N, 2), and bad thresholds; nothing is written"""
    dev = _gpu()
    stages, tuples = (4,), SMALL
    n = nref.num_weights(tuples)
    m, h = 64, 2
    b = torch.zeros((m, 16), dtype=torch.uint8, device=dev)
    target = torch.zeros(m, device=dev)
    ring = torch.zeros((h + 1, m, 16), dtype=torch.uint8, device=dev)
    rew = torch.zeros((h + 1, m), device=dev)
    end = torch.zeros((h + 1, m), dtype=torch.uint8, device=dev)

    def calls(w, coh, acc, st):
        return {
            "value": lambda: ops.ntuple_value(b, w, tuples, stages=st),
            "greedy": lambda: ops.ntuple_greedy(b, w, tuples, stages=st),
            "expectimax": lambda: ops.ntuple_expectimax(b, w, tuples, stages=st),
            "td": lambda: ops.ntuple_td_update(b, target, w, tuples, alpha=0.1, stages=st),
            "tc": lambda: ops.ntuple_tc_update(b, target, w, coh, acc, tuples, alpha=0.1, stages=st),
            "lambda_td": lambda: ops.ntuple_td_lambda_update(ring, rew, end, 0, w, tuples, alpha=0.1, lam=0.5, stages=st),
            "lambda_tc": lambda: ops.ntuple_tc_lambda_update(ring, rew, end, 0, w, coh, acc, tuples, alpha=0.1, lam=0.5,
                                                            stages=st),
        }

    good = (torch.ones(2 * n, device=dev), torch.zeros((2 * n, 2), device=dev), torch.zeros((2 * n, 2), device=dev))
    for size in (n, 3 * n):  # weights of the wrong size for S = 2
        w = torch.ones(size, device=dev)
        for name, call in calls(w, *good[1:], stages).items():
            with pytest.raises(ValueError, match="entries"):
                call()
        assert bool((w == 1).all()), "weights written by a refused call"
    for bad in ((n, 2), (3 * n, 2)):  # coherence, then accum, of the wrong size
        for which in (1, 2):
            args = list(good)
            args[which] = torch.zeros(bad, device=dev)
            for name in ("tc", "lambda_tc"):
                with pytest.raises(ValueError, match="coherence|accum"):
                    calls(*args, stages)[name]()
    for bad in ((5, 4), (4, 4), (0,), (16,), tuple(range(1, 9)), (4.0,), (True,)):
        for name, call in calls(*good, bad).items():
            with pytest.raises(ValueError, match="stage"):
                call()
    assert bool((good[0] == 1).all()) and not bool(good[1].any()) and not bool(good[2].any())
    # the same arguments with the right sizes and thresholds are accepted
    for name, call in calls(*good, stages).items():
        call()
    torch.cuda.synchronize()


# ---- S = 1 and the single-stage entries --------------------------------------------------------------------


def _net_arrays(tuples):
    cells = np.zeros((len(tuples), 6), np.uint8)
    for i, t in enumerate(tuples):
        cells[i, :len(t)] = t
    return cells, np.array([len(t) for t in tuples], np.uint8)


@pytest.mark.gpu
def test_one_stage_equals_the_single_stage_entries(ops, played):
    """stages=() through ops, an explicit S = 1 call of each staged entry through ctypes, and the old entry: bit for bit"""
    from ml2048_b200 import _lib

    lib = _lib.load()
    dev = _gpu()
    rng = np.random.default_rng(50)
    tuples = SMALL
    cells, lens = _net_arrays(tuples)
    c, ln, k = cells.ctypes.data, lens.ctypes.data, len(tuples)
    n = nref.num_weights(tuples)
    boards = torch.from_numpy(np.concatenate([played, _edge_boards(rng, (4, 8))])).to(dev)
    m = boards.shape[0]
    st = ops._stream(boards)
    w0 = torch.from_numpy((rng.standard_normal(n) * 100).astype(np.float32)).to(dev)
    p = lambda t: t.data_ptr()  # noqa: E731

    def bits(t):
        return t.view(torch.int32) if t.dtype == torch.float32 else t

    # value
    outs = [torch.empty(m, device=dev) for _ in range(3)]
    ops.ntuple_value(boards, w0, tuples, out=outs[0])
    assert lib.ml2048_staged_value(p(boards), p(w0), n, c, ln, k, None, 1, p(outs[1]), m, st) == 0
    assert lib.ml2048_ntuple_value(p(boards), p(w0), n, c, ln, k, p(outs[2]), m, st) == 0
    assert torch.equal(bits(outs[0]), bits(outs[1])) and torch.equal(bits(outs[0]), bits(outs[2]))
    # greedy and expectimax (depth 1 and 2 on a few boards)
    def move_outs(q: bool):
        o = {"action": torch.empty(m, dtype=torch.int64, device=dev), "state": torch.empty((m, 16), dtype=torch.uint8, device=dev),
             "reward": torch.empty(m, device=dev), "value": torch.empty(m, device=dev)}
        if q:
            o["q"] = torch.empty((m, 4), device=dev)
        return o

    g = [move_outs(False) for _ in range(3)]
    ops.ntuple_greedy(boards, w0, tuples, reward_fn="improved", out=g[0])
    for j, fn in ((1, lambda *a: lib.ml2048_staged_greedy(*a[:6], None, 1, *a[6:])), (2, lib.ml2048_ntuple_greedy)):
        o = g[j]
        assert fn(p(boards), p(w0), n, c, ln, k, 1, None, p(o["action"]), p(o["state"]), p(o["reward"]), p(o["value"]), m, st) == 0
    for j in (1, 2):
        for key in g[0]:
            assert torch.equal(bits(g[0][key]), bits(g[j][key])), key
    for depth in (1, 2):
        sub = boards[:64] if depth == 2 else boards
        ms = sub.shape[0]
        x = [{kk: v[:ms] for kk, v in move_outs(True).items()} for _ in range(3)]
        ops.ntuple_expectimax(sub, w0, tuples, depth=depth, two_prob=0.9, reward_fn="rank", out=x[0])
        for j, fn in ((1, lambda *a: lib.ml2048_staged_expectimax(*a[:6], None, 1, *a[6:])), (2, lib.ml2048_expectimax)):
            o = x[j]
            assert fn(p(sub), p(w0), n, c, ln, k, 2, depth, 0.9, None, p(o["action"]), p(o["state"]), p(o["reward"]), p(o["value"]),
                      p(o["q"]), ms, st) == 0
        for j in (1, 2):
            for key in x[0]:
                assert torch.equal(bits(x[0][key]), bits(x[j][key])), (depth, key)
    # the four updates from the same start: weights (TC's too: every sum is exact here), coherence and delta
    wi = torch.from_numpy(rng.integers(-8, 9, size=n).astype(np.float32)).to(dev)
    target = torch.from_numpy(rng.integers(-64, 65, size=m).astype(np.float32)).to(dev)
    mask = torch.from_numpy((rng.random(m) < 0.8).astype(np.uint8)).to(dev)
    h = 3
    ring = boards[torch.from_numpy(rng.integers(0, m, size=(h + 1, m))).to(dev)].contiguous()
    rew = torch.from_numpy(rng.choice(np.array([0, 4, 8], np.float32), size=(h + 1, m))).to(dev)
    ended = torch.from_numpy((rng.random((h + 1, m)) < 0.1).astype(np.uint8)).to(dev)
    for rule in ("td", "tc", "lambda_td", "lambda_tc"):
        res = []
        for way in range(3):
            w = wi.clone()
            coh = torch.zeros((n, 2), device=dev)
            acc = torch.zeros((n, 2), device=dev)
            d = torch.empty(m, device=dev)
            tc = (p(coh), p(acc)) if rule.endswith("tc") else ()
            if rule in ("td", "tc"):
                if way == 0:
                    (ops.ntuple_td_update(boards, target, w, tuples, alpha=0.0625, mask=mask, delta_out=d) if rule == "td" else
                     ops.ntuple_tc_update(boards, target, w, coh, acc, tuples, alpha=0.0625, mask=mask, delta_out=d))
                else:
                    head = (p(boards), p(target), p(mask), 0.0625, p(w), *tc, n, c, ln, k)
                    fn = {("td", 1): lib.ml2048_staged_td_update, ("tc", 1): lib.ml2048_staged_tc_update,
                          ("td", 2): lib.ml2048_ntuple_td_update, ("tc", 2): lib.ml2048_tc_update}[(rule, way)]
                    assert fn(*head, *((None, 1) if way == 1 else ()), p(d), m, st) == 0
            else:
                if way == 0:
                    fn = ops.ntuple_td_lambda_update if rule == "lambda_td" else ops.ntuple_tc_lambda_update
                    extra = (w,) if rule == "lambda_td" else (w, coh, acc)
                    fn(ring, rew, ended, 2, *extra, tuples, alpha=0.0625, lam=0.5, mask=mask, delta_out=d)
                else:
                    head = (p(ring), p(rew), p(ended), h, 2, 0.5, p(mask), 0.0625, p(w), *tc, n, c, ln, k)
                    fn = {("lambda_td", 1): lib.ml2048_staged_lambda_td_update, ("lambda_tc", 1): lib.ml2048_staged_lambda_tc_update,
                          ("lambda_td", 2): lib.ml2048_lambda_td_update, ("lambda_tc", 2): lib.ml2048_lambda_tc_update}[(rule, way)]
                    assert fn(*head, *((None, 1) if way == 1 else ()), p(d), m, st) == 0
            torch.cuda.synchronize()
            res.append((w, coh, d))
        for j in (1, 2):
            for a, b in zip(res[0], res[j]):
                assert torch.equal(bits(a), bits(b)), rule
        assert not torch.equal(res[0][0], wi), rule


# ---- CUDA graphs ------------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["td0", "tc", "lambda"])
def test_graph_replay_equals_eager(ops, played, rule):
    """one staged learner step -- greedy on the boards, then the update of the previous afterstates -- captured once and
    replayed on new boards, against the same calls made eagerly from the same start.  Every replay starts from the same
    integer weights and zero coherence (beta = 1), played boards keep rewards and values small, and alpha = 1/64: every delta
    and every sum of deltas is exact in float32, so the order of the atomics cannot change a bit."""
    dev = _gpu()
    stages, tuples = CASES["s3"]
    rng = np.random.default_rng(60)
    m, h = 2048, 3
    n = sref.num_weights(tuples, stages)
    w_init = torch.from_numpy(_stage_weights(rng, tuples, stages, integer=True)).to(dev)
    w = w_init.clone()
    coh = torch.zeros((n, 2), device=dev)
    acc = torch.zeros((n, 2), device=dev)
    s_board = torch.zeros((m, 16), dtype=torch.uint8, device=dev)
    s_prev = torch.zeros((m, 16), dtype=torch.uint8, device=dev)
    s_ring = torch.zeros((h + 1, m, 16), dtype=torch.uint8, device=dev)
    s_rew = torch.zeros((h + 1, m), device=dev)
    s_end = torch.zeros((h + 1, m), dtype=torch.uint8, device=dev)
    target = torch.zeros(m, device=dev)
    d_out = torch.zeros(m, device=dev)
    g_out = {"action": torch.zeros(m, dtype=torch.uint8, device=dev), "state": torch.zeros((m, 16), dtype=torch.uint8, device=dev),
             "reward": torch.zeros(m, device=dev), "value": torch.zeros(m, device=dev)}

    def step(w, coh, acc, board, prev, ring, rew, end, out, d):
        g = ops.ntuple_greedy(board, w, tuples, reward_fn="normal", action_dtype=torch.uint8, out=out, stages=stages)
        if rule == "lambda":
            ops.ntuple_td_lambda_update(ring, rew, end, 2, w, tuples, alpha=0.015625, lam=0.5, delta_out=d, stages=stages)
            return
        torch.add(g["reward"], g["value"], out=target)
        if rule == "td0":
            ops.ntuple_td_update(prev, target, w, tuples, alpha=0.015625, delta_out=d, stages=stages)
        else:
            ops.ntuple_tc_update(prev, target, w, coh, acc, tuples, alpha=0.015625, delta_out=d, stages=stages)

    pool = played
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):  # warm-up outside the capture
        step(w.clone(), coh.clone(), acc, s_board, s_prev, s_ring, s_rew, s_end, {k: v.clone() for k, v in g_out.items()}, d_out.clone())
    torch.cuda.current_stream().wait_stream(stream)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step(w, coh, acc, s_board, s_prev, s_ring, s_rew, s_end, g_out, d_out)
    for _ in range(3):
        s_board.copy_(torch.from_numpy(pool[rng.integers(0, pool.shape[0], size=m)]))
        s_prev.copy_(torch.from_numpy(pool[rng.integers(0, pool.shape[0], size=m)]))
        s_ring.copy_(torch.from_numpy(pool[rng.integers(0, pool.shape[0], size=(h + 1, m))]))
        s_rew.copy_(torch.from_numpy(rng.choice(np.array([0, 4, 8, 256], np.float32), size=(h + 1, m))))
        s_end.copy_(torch.from_numpy((rng.random((h + 1, m)) < 0.1).astype(np.uint8)))
        w.copy_(w_init)
        coh.zero_()
        w_e, c_e = w.clone(), coh.clone()
        inputs = [t.clone() for t in (s_board, s_prev, s_ring, s_rew, s_end)]
        graph.replay()
        e_out = {k: torch.empty_like(v) for k, v in g_out.items()}
        d_e = torch.empty_like(d_out)
        step(w_e, c_e, acc, *inputs, e_out, d_e)
        torch.cuda.synchronize()
        for k in g_out:
            assert torch.equal(g_out[k].view(torch.uint8), e_out[k].view(torch.uint8)), k
        assert torch.equal(d_out.view(torch.int32), d_e.view(torch.int32))
        assert torch.equal(w.view(torch.int32), w_e.view(torch.int32)) and not torch.equal(w, w_init)
        assert torch.equal(coh.view(torch.int32), c_e.view(torch.int32))
        assert not bool(acc.view(torch.int32).any())


# ---- the network, the learner and the policies ------------------------------------------------------------


@pytest.mark.gpu
def test_learner_on_a_staged_network(ops):
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner

    dev = _gpu()
    net = NTupleNetwork(device=dev, stages=(4,))
    n = nref.num_weights(net.tuples)
    assert net.weights.numel() == 2 * n and net.stages == (4,)
    env = VecGame(64, output="torch", sync_free=True, rng_mode="philox")
    learner = TDAfterstateLearner(env, net)
    learner.reset(5)
    reached = False  # some updated afterstate (a masked-in x_0) has a 16 tile
    for _ in range(200):
        prev = learner._prev_after[learner._has_prev.bool()]
        reached = reached or bool((prev.to(torch.int32).amax(dim=1) >= 4).any()) if prev.numel() else reached
        learner.step()
        torch.cuda.synchronize()
        if not reached:
            assert not bool(net.weights[n:].any()), "stage-1 entries written before any afterstate reached a 16 tile"
    assert reached and bool(net.weights[n:].any()) and bool(net.weights[:n].any())
    # every rule runs for a few thousand steps and stays finite; state_dict round trips
    for rule, horizon in (("td0", 1), ("tc", 1), ("td0", 3)):
        net = NTupleNetwork(device=dev, stages=(4,))
        env = VecGame(4096, output="torch", sync_free=True, rng_mode="philox")
        learner = TDAfterstateLearner(env, net, rule=rule, horizon=horizon, lam=0.25)
        learner.reset(7)
        for _ in range(3000):
            learner.step()
        torch.cuda.synchronize()
        assert bool(torch.isfinite(net.weights).all()), rule
        assert bool(net.weights[n:].any()), rule
        sd = net.state_dict()
        assert sd["stages"] == [4]
        other = NTupleNetwork(device=dev, stages=[4])
        other.load_state_dict(sd)
        assert torch.equal(other.weights, net.weights)
        if rule == "tc":
            assert other.coherence.shape == (2 * n, 2) and torch.equal(other.coherence, net.coherence)
        with pytest.raises(ValueError):
            NTupleNetwork(device=dev).load_state_dict(sd)
        with pytest.raises(ValueError):
            NTupleNetwork(device=dev, stages=(5,)).load_state_dict(sd)
    # an old dict without "stages" is a single-stage network's
    single = NTupleNetwork(SMALL, device=dev)
    single.weights.copy_(torch.randn(single.weights.numel(), device=dev))
    old = single.state_dict()
    del old["stages"]
    fresh = NTupleNetwork(SMALL, device=dev)
    fresh.load_state_dict(old)
    assert torch.equal(fresh.weights, single.weights)
    with pytest.raises(ValueError):
        NTupleNetwork(SMALL, device=dev, stages=(4,)).load_state_dict(old)


@pytest.mark.gpu
def test_policies_under_device_runner(ops):
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import ExpectimaxPolicy, GreedyPolicy, NTupleNetwork
    from ml2048_b200.runner import DeviceRunner

    dev = _gpu()
    net = NTupleNetwork(SMALL, device=dev, stages=(3, 5))
    net.weights.copy_(torch.randn(net.weights.numel(), device=dev) * 100)
    env = VecGame(512, "improved", two_prob=0.7, output="torch", sync_free=True)
    env.reset(1)
    for name, pol in (("greedy", GreedyPolicy(net, reward_fn="improved")),
                      ("expectimax1", ExpectimaxPolicy(net, depth=1, reward_fn="improved", two_prob=0.7)),
                      ("expectimax2", ExpectimaxPolicy(net, depth=2, reward_fn="improved", two_prob=0.7))):
        runner = DeviceRunner(env, 512)
        seen = []
        runner.add_callback("prepared", lambda e, idx: seen.append(("board", e.observations()[0].clone())))
        runner.add_callback("stepped", lambda e, res, actions, lp: seen.append(("action", actions.clone(), lp.clone())))
        for _ in range(6):
            runner.step_once(pol)
        assert len(seen) == 12
        for (_, board), (_, actions, lp) in zip(seen[0::2], seen[1::2]):
            if name == "greedy":
                want = ops.ntuple_greedy(board, net.weights, net.tuples, reward_fn="improved", stages=net.stages)["action"]
            else:
                want = ops.ntuple_expectimax(board, net.weights, net.tuples, depth=int(name[-1]), two_prob=0.7, reward_fn="improved",
                                             stages=net.stages)["action"]
            assert torch.equal(actions.to(dev), want) and not bool(lp.any()), name
