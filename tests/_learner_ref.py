"""Plain restatement of ml2048_b200.ntuple.TDAfterstateLearner over the C oracle (oracle.OracleVecGame), for the tests.

Built only from the op references (_ntuple_ref, _tc_ref, _lambda_ref, _stage_ref, _promotion_ref) and the oracle's moves
(_expectimax_ref.oracle_move).  The learner's state is its own: the previous afterstate, whether its game ended, whether
there is one, the ring of the last h + 1 afterstates, rewards and end flags, and the step count since reset().  The
weights W, the TC coherence C and the promotion marks P are not state here: each step takes them as arguments, so that a
caller can hand it the device's values before every step.  One step:

  1. prepare(); the boards.
  2. For every board its four afterstates, rewards and validity from the oracle; the greedy action, afterstate, reward and
     value on W (and P).
  3. The update:
     h = 1: x_0 is the previous afterstate, the target reward + value of the move just chosen (one float32 add), 0 where
            x_0's game ended; games without a previous afterstate (the first step after reset()) are masked out.
     h > 1: the greedy afterstate and reward go into slot T mod (h + 1) (T = steps since reset()).  Steps 0 .. h-1 update
            nothing; from step h on, every game's x_0 = the afterstate of step T - h is updated toward the lambda-return
            of its window, truncated at the first end in it.
     With alpha = 0 there is no update at all.  The expected result: delta bit for bit, the marks and the promoted copies
     exactly, and the weights and coherence in float64 with the adds per entry and sum |delta| per entry that bound the
     float32 atomics.
  4. step(action); the end flags are recorded (h = 1: for the next target; h > 1: in the ring's slot of this step).
reset(seed) restarts the games and drops the pending update and the window.
"""

from __future__ import annotations

from typing import Optional

import numpy as np

import _expectimax_ref as xref
import _lambda_ref as lref
import _ntuple_ref as nref
import _promotion_ref as pref
import _stage_ref as sref
import _tc_ref as tref

RESULT_KEYS = ("state", "valid_actions", "merged", "step", "reward", "score", "terminated", "invalid", "prev_state",
               "prev_valid_actions")


class RefLearner:
    """``form``: which op references state the network: "single" (_ntuple_ref / _tc_ref / _lambda_ref), "staged"
    (_stage_ref) or "promoted" (_promotion_ref); by default "promoted" with ``promotion``, "staged" with stages, else
    "single".  ``window``: run the ring form of step 3 (by default h > 1)."""

    def __init__(self, oracle, m: int, kind: str, two_prob: float, tuples, *, stages=(), promotion: bool = False,
                 rule: str = "td0", horizon: int = 1, lam: float = 0.5, alpha: float, form: Optional[str] = None,
                 window: Optional[bool] = None):
        assert rule in ("td0", "tc") and horizon >= 1
        self.env = oracle.OracleVecGame(m, kind, two_prob=two_prob)
        self.move = xref.oracle_move(oracle, kind)
        self.m, self.tuples, self.stages = m, tuple(tuple(t) for t in tuples), tuple(stages)
        self.form = form or ("promoted" if promotion else "staged" if stages else "single")
        self.rule, self.h, self.lam, self.alpha = rule, horizon, lam, float(alpha)
        self.window = horizon > 1 if window is None else window
        self.prev_after = np.zeros((m, 16), np.uint8)
        self.prev_ended = np.zeros(m, bool)
        self.has_prev = np.zeros(m, bool)
        self.ring_after = np.zeros((horizon + 1, m, 16), np.uint8)
        self.ring_reward = np.zeros((horizon + 1, m), np.float32)
        self.ring_ended = np.zeros((horizon + 1, m), np.uint8)
        self.steps = 0
        self.delta = np.zeros(m, np.float32)

    def reset(self, seed: int) -> None:
        self.env.reset(seed)
        self.has_prev[:] = False
        self.steps = 0
        self.delta = np.zeros(self.m, np.float32)

    # ---- the network, through the references of its form --------------------------------------------------------------

    def _read_weights(self, w, p):
        """the weights every read uses: the effective weights of a promoting network"""
        return pref.effective(w, p, self.tuples, self.stages) if self.form == "promoted" else w

    def _greedy(self, board, w, p) -> dict:
        after, reward, valid = self.move(board)
        if self.form == "single":
            return nref.greedy(board, after, reward, valid, w, self.tuples)
        if self.form == "staged":
            return sref.greedy(board, after, reward, valid, w, self.tuples, self.stages)
        return pref.greedy(board, after, reward, valid, w, p, self.tuples, self.stages)

    def _td_delta(self, x0, target, w, p, mask):
        if self.form == "single":
            return nref.td_delta(x0, target, w, self.tuples, self.alpha, mask)
        return sref.td_delta(x0, target, self._read_weights(w, p), self.tuples, self.stages, self.alpha, mask)

    def _ring_delta(self, newest, w, p):
        ring = (self.ring_after, self.ring_reward, self.ring_ended, newest)
        if self.form == "single":
            return lref.ring_delta(*ring, w, self.tuples, self.lam, self.alpha)
        return sref.ring_delta(*ring, self._read_weights(w, p), self.tuples, self.stages, self.lam, self.alpha)

    def _apply(self, x0, d, mask, w, c, p) -> dict:
        """promotion (a promoting network), then the float64 apply of the rule"""
        tc = self.rule == "tc"
        w0, c0, marks = np.array(w, np.float32), None if c is None else np.array(c, np.float32), None
        if self.form == "promoted":
            w0, marks, c0 = pref.promote(x0, w, p, self.tuples, self.stages, mask, c if tc else None)
            if not tc:
                c0 = None if c is None else np.array(c, np.float32)
        out = {"x0": x0, "delta": d, "mask": mask, "w0": w0, "c0": c0, "marks": marks}
        if tc:
            if self.form == "single":
                w64, e64, a64, adds, sabs = tref.tc_apply_f64(x0, d, w0, c0, self.tuples, mask)
            else:
                w64, e64, a64, adds, sabs = sref.tc_apply_f64(x0, d, w0, c0, self.tuples, self.stages, mask)
            out.update(w64=w64, e64=e64, a64=a64, adds=adds, sabs=sabs)
        else:
            if self.form == "single":
                w64, adds, sabs = nref.td_apply_f64(x0, d, w0, self.tuples, mask)
            else:
                w64, adds, sabs = sref.td_apply_f64(x0, d, w0, self.tuples, self.stages, mask)
            out.update(w64=w64, adds=adds, sabs=sabs)
        return out

    # ---- one learner step ------------------------------------------------------------------------------------------

    def step(self, weights, coherence=None, promoted=None) -> dict:
        """one step from W = ``weights``, C = ``coherence`` ((S * N, 2); None reads as zeros) and P = ``promoted``:
        {"board", "action", "afterstate", "reward", "value", "delta", "update" (None when nothing is updated, else the
        expected update, see _apply), "result" (the step's fields, copies)}"""
        w = np.asarray(weights, np.float32)
        c = coherence
        if self.rule == "tc" and c is None:
            c = np.zeros((w.size, 2), np.float32)
        env = self.env
        env.prepare()
        board = env.observations()[0].copy()
        g = self._greedy(board, w, promoted)
        update = None
        if not self.window:
            if self.alpha != 0.0:
                target = np.where(self.prev_ended, np.float32(0), (g["reward"] + g["value"]).astype(np.float32))
                mask = self.has_prev.copy()
                self.delta = self._td_delta(self.prev_after, target.astype(np.float32), w, promoted, mask)
                update = self._apply(self.prev_after.copy(), self.delta, mask, w, c, promoted)
        else:
            newest = self.steps % (self.h + 1)
            self.ring_after[newest] = g["state"]
            self.ring_reward[newest] = g["reward"]
            if self.alpha != 0.0 and self.steps >= self.h:
                self.delta, x0 = self._ring_delta(newest, w, promoted)
                update = self._apply(x0.copy(), self.delta, np.ones(self.m, bool), w, c, promoted)
        res = env.step(np.asarray(g["action"], np.int64))
        result = {k: np.array(res[k]) for k in RESULT_KEYS}
        ended = result["terminated"] != 0
        if not self.window:
            self.prev_after = np.array(g["state"], np.uint8)
            self.prev_ended = ended
            self.has_prev[:] = True
        else:
            self.ring_ended[newest] = ended
            self.steps += 1
        return {"board": board, "action": np.asarray(g["action"], np.int64), "afterstate": np.array(g["state"], np.uint8),
                "reward": g["reward"], "value": g["value"], "delta": self.delta.copy(), "update": update, "result": result}
