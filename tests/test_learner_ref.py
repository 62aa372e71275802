"""
The reference learner (tests/_learner_ref.py) against plain per-game Python loops over the C oracle, on the CPU.

- Every rule (TD(0), TC, TD(lambda) h = 3, TC(lambda) h = 2) on a single-stage, a staged and a promoting network, M = 6
  games for 120 steps from one seed, with a reset(seed) in the middle: the greedy action, afterstate, reward and value and
  every field of the step bit for bit; delta bit for bit; the expected weights, coherence, adds per entry and sum |delta|
  per entry against a game-by-game float64 loop; the marks and the promoted copies exactly.  Games end inside the run, and
  the updated afterstates cover every stage.
- Identities: h = 1 through the ring equals the TD(0) / TC form; form "staged" with S = 1 equals "single"; a promoting
  network whose every mark is set equals the staged network and leaves the marks; alpha = 0 updates nothing and plays the
  greedy policy's game.
"""

from __future__ import annotations

import numpy as np
import pytest

import _learner_ref as lr

TUPLES = ((0, 1, 2), (4, 5, 6), (0, 4, 8), (1, 5, 9, 13))
STAGES = (3, 5)
KINDS = ("normal", "improved", "rank", "maxcell")

# ---- the brute force: one game at a time -----------------------------------------------------------------------------


def _images(b: np.ndarray) -> np.ndarray:
    """the 8 symmetric images of one board, (8, 16): image g holds in (r, c) the cell (r, c), (r, 3-c), (3-r, c),
    (3-r, 3-c), (c, r), (c, 3-r), (3-c, r), (3-c, 3-r) of b"""
    g = b.reshape(4, 4)
    t = g.T
    return np.stack([g, g[:, ::-1], g[::-1, :], g[::-1, ::-1], t, t[::-1, :], t[:, ::-1], t[::-1, ::-1]]).reshape(8, 16)


class Brute:
    def __init__(self, tuples, stages, promotion):
        self.tuples, self.stages, self.promotion = tuples, stages, promotion
        self.n = sum(16 ** len(t) for t in tuples)
        self.offs = [sum(16 ** len(u) for u in tuples[:i]) for i in range(len(tuples))]

    def stage(self, b) -> int:
        top = max(min(int(x), 15) for x in b)
        return sum(1 for tau in self.stages if tau <= top)

    def entries(self, b):
        """(stage, [single-stage entry of tuple t, image g for t, g in order])"""
        img = _images(np.asarray(b))
        out = []
        for t, cells in enumerate(self.tuples):
            for g in range(8):
                out.append(self.offs[t] + sum(min(int(img[g][c]), 15) << (4 * j) for j, c in enumerate(cells)))
        return self.stage(b), out

    def read(self, w, p, s: int, e: int) -> np.float32:
        if self.promotion:
            while s >= 1 and not (int(p[e]) >> (s - 1)) & 1:
                s -= 1
        return w[s * self.n + e]

    def value(self, b, w, p) -> np.float32:
        s, ents = self.entries(b)
        acc = np.float32(0)
        for e in ents:
            acc = np.float32(acc + self.read(w, p, s, e))
        return acc

    def greedy(self, oracle, kind, b, w, p):
        best, bkey = None, None
        for a in range(4):
            nb, mg = oracle.board_move(b, a)
            if not (nb != b).any():
                continue
            r = np.float32(oracle.board_reward(kind, nb, b, mg))
            v = self.value(nb, w, p)
            q = np.float32(r + v)
            key = np.float32(-np.inf) if np.isnan(q) else q
            if best is None or key > bkey:
                best, bkey = (a, nb, r, v), key
        return best if best is not None else (0, np.array(b), np.float32(0), np.float32(0))

    def apply(self, updates, w, c, p, rule):
        """updates: [(x0, delta)] of the masked-in games in game order -> w0, c0, marks, w64, e64, a64, adds, sabs"""
        w0 = np.array(w, np.float32)
        c0 = None if c is None else np.array(c, np.float32)
        marks = None if p is None else np.array(p, np.uint8)
        if self.promotion:
            before_w, before_p = np.array(w, np.float32), np.array(p, np.uint8)
            for x0, _ in updates:
                s0, ents = self.entries(x0)
                if s0 == 0:
                    continue
                for e in ents:
                    if not (int(before_p[e]) >> (s0 - 1)) & 1:
                        w0[s0 * self.n + e] = self.read(before_w, before_p, s0 - 1, e)
                        if rule == "tc":
                            c0[s0 * self.n + e] = 0.0
                        marks[e] |= 1 << (s0 - 1)
        size = w0.size
        de, sabs, adds = np.zeros(size), np.zeros(size), np.zeros(size, np.int64)
        for x0, d in updates:
            s0, ents = self.entries(x0)
            for e in ents:
                j = s0 * self.n + e
                de[j] += float(d)
                sabs[j] += abs(float(d))
                adds[j] += 1
        out = {"w0": w0, "c0": c0, "marks": marks, "adds": adds, "sabs": sabs}
        if rule == "td0":
            out["w64"] = w0.astype(np.float64) + de
            return out
        w64, e64, a64 = w0.astype(np.float64), c0[:, 0].astype(np.float64), c0[:, 1].astype(np.float64)
        for j in np.flatnonzero(sabs):
            e_0, a_0 = c0[j]
            beta = 1.0 if a_0 == 0 else float(np.float32(np.float32(abs(e_0)) / a_0))
            w64[j] += beta * de[j]
            e64[j] += de[j]
            a64[j] += sabs[j]
        out.update(w64=w64, e64=e64, a64=a64)
        return out


class BruteLearner:
    """TDAfterstateLearner's step restated game by game"""

    def __init__(self, oracle, m, kind, two_prob, tuples, stages, promotion, rule, h, lam, alpha):
        self.oracle, self.kind = oracle, kind
        self.env = oracle.OracleVecGame(m, kind, two_prob=two_prob)
        self.net = Brute(tuples, stages, promotion)
        self.m, self.rule, self.h, self.alpha = m, rule, h, np.float32(alpha)
        self.lf = np.float32(lam)
        self.c = np.float32(np.float32(1) - self.lf)

    def reset(self, seed):
        self.env.reset(seed)
        self.prev = [None] * self.m  # (afterstate, ended) of the previous step, per game
        self.hist = [[] for _ in range(self.m)]  # [afterstate, reward, ended] of every step since reset, per game
        self.delta = np.zeros(self.m, np.float32)

    def _lambda_delta(self, win, w, p):
        """win: the last h + 1 [afterstate, reward, ended] of one game, oldest first"""
        h, net = self.h, self.net
        v = [net.value(x, w, p) for x, _, _ in win]
        r = np.float32(0) if win[h - 1][2] else np.float32(win[h][1] + v[h])
        for k in range(h - 2, -1, -1):
            if win[k][2]:
                r = np.float32(0)
            else:
                r = np.float32(np.float32(win[k + 1][1] + np.float32(self.c * v[k + 1])) + np.float32(self.lf * r))
        return np.float32(self.alpha * np.float32(r - v[0]))

    def step(self, w, c, p):
        env, net = self.env, self.net
        if self.rule == "tc" and c is None:
            c = np.zeros((np.asarray(w).size, 2), np.float32)
        env.prepare()
        boards = env.observations()[0].copy()
        chosen = [net.greedy(self.oracle, self.kind, b, w, p) for b in boards]
        updates = None
        if self.h == 1:
            if self.alpha != 0:
                updates = []
                for i, (_, after, r, v) in enumerate(chosen):
                    if self.prev[i] is None:
                        self.delta[i] = 0.0
                        continue
                    x0, ended = self.prev[i]
                    target = np.float32(0) if ended else np.float32(r + v)
                    self.delta[i] = np.float32(self.alpha * np.float32(target - net.value(x0, w, p)))
                    updates.append((x0, self.delta[i]))
        else:
            for i, (_, after, r, _) in enumerate(chosen):
                self.hist[i].append([after, r, False])
            if self.alpha != 0 and len(self.hist[0]) > self.h:
                updates = []
                for i in range(self.m):
                    win = self.hist[i][-(self.h + 1):]
                    self.delta[i] = self._lambda_delta(win, w, p)
                    updates.append((win[0][0], self.delta[i]))
        res = env.step(np.array([a for a, _, _, _ in chosen], np.int64))
        for i, (_, after, _, _) in enumerate(chosen):
            ended = bool(res["terminated"][i])
            if self.h == 1:
                self.prev[i] = (after, ended)
            else:
                self.hist[i][-1][2] = ended
        return {"chosen": chosen, "delta": self.delta.copy(), "result": {k: np.array(res[k]) for k in lr.RESULT_KEYS},
                "update": None if updates is None else net.apply(updates, w, c, p, self.rule)}


# ---- helpers ----------------------------------------------------------------------------------------------------


def _start(rng, tuples, stages, promotion, scale=4.0):
    """random weights of every stage; for a promoting network clear marks and NaN in the storage they hide"""
    n = sum(16 ** len(t) for t in tuples)
    s = len(stages) + 1
    w = (rng.standard_normal(s * n) * scale).astype(np.float32)
    p = np.zeros(n, np.uint8) if promotion else None
    if promotion:
        w[n:] = np.nan
    return w, p


def _bits(a, b, what):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    np.testing.assert_array_equal(np.isnan(a), np.isnan(b), err_msg=what)
    np.testing.assert_array_equal(a[~np.isnan(a)].view(np.uint32), b[~np.isnan(b)].view(np.uint32), err_msg=what)


def _crowd(oracle, env) -> None:
    """games 0 and 1 continue from a board with one empty cell and no pair whatever the spawn: they end in the next step"""
    b = np.array([0, 3, 4, 5, 6, 7, 8, 9, 3, 4, 5, 6, 7, 8, 9, 10], np.uint8)
    d = env._data
    for i in (0, 1):
        d["board"][i] = b
        d["valid_actions"][i] = oracle.board_valid(b)
        d["terminated"][i] = 0


def _next_state(upd, w, c, p):
    """the float32 weights, coherence and marks to feed the next step: the float64 result rounded"""
    if upd is None:
        return w, c, p
    c2 = None if "e64" not in upd else np.stack([upd["e64"], upd["a64"]], axis=1).astype(np.float32)
    return upd["w64"].astype(np.float32), c2 if c2 is not None else c, upd["marks"] if upd["marks"] is not None else p


def _same_update(got, want, exact: bool):
    if want is None:
        assert got is None
        return
    assert got is not None
    _bits(got["w0"], want["w0"], "w0")
    np.testing.assert_array_equal(got["adds"], want["adds"])
    if want["marks"] is None:
        assert got["marks"] is None
    else:
        np.testing.assert_array_equal(got["marks"], want["marks"])
    keys = ("w64", "sabs") + (("e64", "a64") if "e64" in want else ())
    for k in keys:
        if exact:
            np.testing.assert_array_equal(got[k], want[k], err_msg=k)
        else:
            np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=1e-12, err_msg=k)
    if "e64" in want:
        _bits(got["c0"], want["c0"], "c0")


# ---- the reference against the brute force ----------------------------------------------------------------------------

RULES = {"td0": ("td0", 1, 0.5), "tc": ("tc", 1, 0.5), "td_lambda": ("td0", 3, 0.5), "tc_lambda": ("tc", 2, 0.25)}
NETS = {"single": ((), False), "staged": (STAGES, False), "promoted": (STAGES, True)}


@pytest.mark.parametrize("net", list(NETS))
@pytest.mark.parametrize("rule", list(RULES))
def test_reference_learner_against_brute_force(oracle, rule, net):
    i = list(RULES).index(rule) * 3 + list(NETS).index(net)
    kind, two_prob = KINDS[i % 4], (0.8, 0.5, 1.0)[i % 3]
    r, h, lam = RULES[rule]
    stages, promotion = NETS[net]
    m, steps, alpha = 6, 120, 0.05
    rng = np.random.default_rng(10 + i)
    w, p = _start(rng, TUPLES, stages, promotion)
    c = None
    ref = lr.RefLearner(oracle, m, kind, two_prob, TUPLES, stages=stages, promotion=promotion, rule=r, horizon=h, lam=lam,
                        alpha=alpha)
    brute = BruteLearner(oracle, m, kind, two_prob, TUPLES, stages, promotion, r, h, lam, alpha)
    ends, updated_stages, masked_steps = 0, set(), 0
    for t in range(steps):
        if t in (0, 70):
            ref.reset(5 + t)
            brute.reset(5 + t)
            since_reset = 0
        got = ref.step(w, c, p)
        want = brute.step(w, c, p)
        np.testing.assert_array_equal(got["action"], [x[0] for x in want["chosen"]])
        np.testing.assert_array_equal(got["afterstate"], np.stack([x[1] for x in want["chosen"]]))
        _bits(got["reward"], [x[2] for x in want["chosen"]], "reward")
        _bits(got["value"], [x[3] for x in want["chosen"]], "value")
        for k in lr.RESULT_KEYS:
            np.testing.assert_array_equal(got["result"][k], want["result"][k], err_msg=k)
        _bits(got["delta"], want["delta"], f"delta at step {t}")
        _same_update(got["update"], want["update"], exact=False)
        if since_reset < h:  # the pending update (h = 1) or the window (h > 1) is empty after reset()
            assert not got["delta"].any() and (got["update"] is None or not got["update"]["adds"].any())
            masked_steps += 1
        elif got["update"] is not None:
            x0 = got["update"]["x0"]
            updated_stages |= set(int(Brute(TUPLES, stages, False).stage(b)) for b in x0)
        since_reset += 1
        ends += int(got["result"]["terminated"].sum())
        w, c, p = _next_state(got["update"], w, c, p)
        if t in (0, 70):
            for env in (ref.env, brute.env):
                _crowd(oracle, env)
    assert ends > 0
    assert masked_steps == 2 * h
    assert updated_stages == set(range(len(stages) + 1)), updated_stages
    if promotion:
        assert p.any() and not np.isnan(w[:sum(16 ** len(x) for x in TUPLES)]).any()


# ---- identities -------------------------------------------------------------------------------------------------


def _lockstep(a, b, w, c, p, steps, exact=True, seed=3):
    a.reset(seed)
    b.reset(seed)
    for _ in range(steps):
        x, y = a.step(w, c, p), b.step(w, c, p)
        for k in ("action", "afterstate"):
            np.testing.assert_array_equal(x[k], y[k])
        for k in lr.RESULT_KEYS:
            np.testing.assert_array_equal(x["result"][k], y["result"][k])
        _bits(x["delta"], y["delta"], "delta")
        yield x, y
        w, c, p = _next_state(x["update"], w, c, p)


def _or_unchanged(upd, w):
    """an update that changes nothing, for a step without one"""
    if upd is not None:
        return upd
    return {"w0": w, "c0": None, "marks": None, "adds": np.zeros(w.size, np.int64), "w64": w.astype(np.float64),
            "sabs": np.zeros(w.size)}


@pytest.mark.parametrize("rule", ["td0", "tc"])
def test_h1_window_equals_td0_and_tc(oracle, rule):
    w, _ = _start(np.random.default_rng(1), TUPLES, (), False)
    kw = dict(rule=rule, horizon=1, alpha=0.05)
    a = lr.RefLearner(oracle, 8, "improved", 0.8, TUPLES, **kw)
    b = lr.RefLearner(oracle, 8, "improved", 0.8, TUPLES, window=True, **kw)
    for x, y in _lockstep(a, b, w, None, None, 60):
        xu, yu = _or_unchanged(x["update"], w), _or_unchanged(y["update"], w)
        np.testing.assert_array_equal(xu["adds"], yu["adds"])
        np.testing.assert_array_equal(xu["w64"], yu["w64"])
        if "e64" in xu and "e64" in yu:
            np.testing.assert_array_equal(xu["e64"], yu["e64"])
            np.testing.assert_array_equal(xu["a64"], yu["a64"])
        w = x["update"]["w64"].astype(np.float32) if x["update"] is not None else w


@pytest.mark.parametrize("rule,h", [("td0", 1), ("tc", 1), ("td0", 3), ("tc", 2)])
def test_one_stage_equals_single_stage(oracle, rule, h):
    w, _ = _start(np.random.default_rng(2), TUPLES, (), False)
    kw = dict(rule=rule, horizon=h, lam=0.25, alpha=0.05)
    a = lr.RefLearner(oracle, 8, "rank", 0.5, TUPLES, **kw)
    b = lr.RefLearner(oracle, 8, "rank", 0.5, TUPLES, form="staged", **kw)
    assert a.form == "single"
    for x, y in _lockstep(a, b, w, None, None, 40):
        _same_update(x["update"], y["update"], exact=True)


@pytest.mark.parametrize("rule,h", [("td0", 1), ("tc", 1), ("td0", 3), ("tc", 2)])
def test_every_mark_set_equals_staged(oracle, rule, h):
    w, _ = _start(np.random.default_rng(3), TUPLES, STAGES, False)
    full = np.full(sum(16 ** len(t) for t in TUPLES), (1 << len(STAGES)) - 1, np.uint8)
    kw = dict(stages=STAGES, rule=rule, horizon=h, lam=0.5, alpha=0.05)
    a = lr.RefLearner(oracle, 8, "maxcell", 1.0, TUPLES, promotion=True, **kw)
    b = lr.RefLearner(oracle, 8, "maxcell", 1.0, TUPLES, **kw)
    steps = 0
    for x, y in _lockstep(a, b, w, None, full, 40):
        if x["update"] is not None:
            np.testing.assert_array_equal(x["update"]["marks"], full)
            x["update"]["marks"] = None
            steps += 1
        _same_update(x["update"], y["update"], exact=True)
    assert steps > 30


def test_alpha_zero_updates_nothing_and_plays_greedy(oracle):
    m = 8
    w, p = _start(np.random.default_rng(4), TUPLES, STAGES, True)
    p[:] = np.random.default_rng(5).integers(0, 4, p.size)
    for rule, h in (("td0", 1), ("tc", 3)):
        ref = lr.RefLearner(oracle, m, "normal", 0.8, TUPLES, stages=STAGES, promotion=True, rule=rule, horizon=h, alpha=0.0)
        brute = BruteLearner(oracle, m, "normal", 0.8, TUPLES, STAGES, True, rule, h, 0.5, 0.0)
        ref.reset(9)
        brute.reset(9)
        for _ in range(50):
            got, want = ref.step(w, None, p), brute.step(w, None, p)
            assert got["update"] is None and want["update"] is None and not got["delta"].any()
            np.testing.assert_array_equal(got["action"], [x[0] for x in want["chosen"]])
            for k in lr.RESULT_KEYS:
                np.testing.assert_array_equal(got["result"][k], want["result"][k], err_msg=k)
