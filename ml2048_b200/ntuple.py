"""N-tuple value networks on the device and a TD(0) afterstate learner over ``VecGame``.

An n-tuple network (Szubert & Jaskowski 2014; Yeh et al. 2016) values a 2048 board as a sum of table entries indexed by the
4-bit fields of a few cells, over the board's 8 symmetric images (one table per tuple, shared by the images).  Evaluating it,
choosing the greedy afterstate move with it and updating it are integer byte work on boards plus scattered 4-byte reads and
adds: each is one kernel here (``ops.ntuple_value``, ``ops.ntuple_greedy``, ``ops.ntuple_td_update``; temporal coherence
learning, a step size per weight, is ``ops.ntuple_tc_update`` and ``TDAfterstateLearner(..., rule="tc")``; their delayed
lambda-return forms are ``ops.ntuple_td_lambda_update`` / ``ntuple_tc_lambda_update`` and ``TDAfterstateLearner(...,
horizon=h, lam=lam)``).  ``NTupleNetwork(..., stages=(tau_1, ...))`` is a multi-stage network (Yeh et al. 2016): one weight
set per stage of the game, chosen by the board's largest tile (``ops.ntuple_stages``); with ``promotion=True`` a stage's entry
starts from the stage below on its first update (Jaskowski 2018).

    net = NTupleNetwork(device="cuda")                        # the standard 4x6 network, zero weights (256 MiB)
    env = VecGame(16384, output="torch", sync_free=True)
    env.reset(0)
    learner = TDAfterstateLearner(env, net)
    for _ in range(n):
        learner.step()                                        # prepare, greedy, TD(0) update of the previous afterstate, step
    env.episode_stats()
"""

from __future__ import annotations

from typing import Any, Optional

import torch

from . import ops

# Szubert & Jaskowski's 4x6 network: two straight 6-tuples (rows 0-1, rows 1-2) and two 2x3 rectangles
STANDARD_4X6 = ((0, 1, 2, 3, 4, 5), (4, 5, 6, 7, 8, 9), (0, 1, 2, 4, 5, 6), (4, 5, 6, 8, 9, 10))

# Step size of TDAfterstateLearner: alpha = DEFAULT_ALPHA_TIMES_GAMES / M.  One call adds the deltas of all M games at once,
# and early-game boards share table entries across a large fraction of the batch, so the summed step on such an entry grows
# with M: a fixed alpha that learns at one batch size diverges to NaN at a larger one.  tools/ntuple_bench.py swept
# alpha = c / M for c = 0.1 ... 3.2 at M = 4096, 2^14 and 2^16, 30 000 steps each (profiles/ntuple_bench.txt, B200): the
# results depend on c alone, not on M (mean score 9.8k / 11.7k / 14.4k / 5.5k / 2.2k / 1.6-2.2k for c = 0.1 / 0.2 / 0.4 /
# 0.8 / 1.6 / 3.2 at all three sizes), and c = 0.4 is the best of them.  Every default step size in this module was swept for
# single-stage networks only: no sweep has been run for multi-stage ones (NTupleNetwork(stages=...)), which use the same
# defaults.
DEFAULT_ALPHA_TIMES_GAMES = 0.4


def default_alpha(num_games: int) -> float:
    return DEFAULT_ALPHA_TIMES_GAMES / num_games


# Step size of TDAfterstateLearner(rule="tc"): alpha = DEFAULT_TC_ALPHA_TIMES_GAMES / M, for the same reason as above (the
# batch sums the steps of all M games on shared entries).  tools/tc_bench.py swept c = 0.1 ... 6.4 at M = 4096, 2^14 and 2^16,
# 30 000 steps each (profiles/tc_bench.txt, B200): again the results depend on c alone (mean score 10.1k / 11.7-11.8k /
# 13.9-14.0k / 16.3-16.4k / 8.5-9.0k / 4.3-4.9k / 4.0-4.9k for c = 0.1 / 0.2 / 0.4 / 0.8 / 1.6 / 3.2 / 6.4 at all three
# sizes), and c = 0.8, twice TD(0)'s best, is the best of them.
DEFAULT_TC_ALPHA_TIMES_GAMES = 0.8


def default_tc_alpha(num_games: int) -> float:
    return DEFAULT_TC_ALPHA_TIMES_GAMES / num_games


# Step size of TDAfterstateLearner(rule="tc", horizon=h > 1): alpha = DEFAULT_TC_LAMBDA_ALPHA_TIMES_GAMES / M.
# tools/lambda_bench.py swept c = 0.2 ... 3.2 at M = 2^14 for the best (h, lambda) = (2, 0.25) of its sweep at c = 0.8, 30 000
# steps each (profiles/lambda_bench.txt, B200): mean score 12.0k / 14.2k / 8.9k / 4.1k / 4.0k for c = 0.2 / 0.4 / 0.8 / 1.6 /
# 3.2, so delayed TC(lambda) takes half of TC's step size.  TD(lambda)'s best c is TD(0)'s 0.4.
DEFAULT_TC_LAMBDA_ALPHA_TIMES_GAMES = 0.4


class NTupleNetwork:
    """An n-tuple value function with its weights on one CUDA device.

    ``tuples``: 1..16 tuples of 1..6 distinct cells (cell = row*4 + col).  The weights are one zero-initialised float32 tensor
    of sum 16^len entries, tuple t's table after those of the tuples before it (``offsets``).

    ``stages``: 0..7 strictly ascending tile exponents tau_1 < ... in 1..15 (``ops.ntuple_stages``) make a multi-stage network
    of S = len(stages) + 1 weight sets.  A board b is in stage #{k : tau_k <= max_c min(b[c], 15)}, and is valued and updated
    with that stage's tables; the weights are S * N entries, stage s's tables at s * N (N = sum 16^len), and ``coherence``
    is (S * N, 2).  ``stages=()`` is the single-stage network.

    ``promotion=True`` (multi-stage only) adds weight promotion (Jaskowski 2018): ``promoted`` is an (N,) uint8 tensor of
    marks, all clear at first, so that every stage >= 1 starts as stage 0.  Each op reads an unwritten entry of stage s
    through stage s - 1, and an update first copies that value into every entry it is about to change (``ops.ntuple_value``,
    ``ops.ntuple_td_update``).  ``promoted`` is None without promotion."""

    def __init__(self, tuples=STANDARD_4X6, device: Any = None, *, stages=(), promotion: bool = False):
        self.tuples = ops.ntuple_spec(tuples)
        self.stages = ops.ntuple_stages(stages)
        if promotion and not self.stages:
            raise ValueError("promotion=True needs a multi-stage network (stages=...)")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.type != "cuda":
            raise ValueError(f"device={device!r}: ml2048_b200 runs on CUDA only")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        self.offsets = []
        total = 0
        for t in self.tuples:
            self.offsets.append(total)
            total += 16 ** len(t)
        self.weights = torch.zeros(((len(self.stages) + 1) * total,), dtype=torch.float32, device=dev)
        self.promoted: Optional[torch.Tensor] = torch.zeros((total,), dtype=torch.uint8, device=dev) if promotion else None
        # TC learning's {E, A} per weight and the TC updates' scratch (all zero between calls), allocated by the first TC update
        self.coherence: Optional[torch.Tensor] = None
        self._tc_accum: Optional[torch.Tensor] = None

    def value(self, board: torch.Tensor, *, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """V of (M,16) boards: (M,) float32 (``ops.ntuple_value``)."""
        return ops.ntuple_value(board, self.weights, self.tuples, out=out, stages=self.stages, promoted=self.promoted)

    def greedy(self, board: torch.Tensor, *, reward_fn=None, action_dtype: torch.dtype = torch.int64,
               out: Optional[dict] = None) -> dict:
        """The move maximising reward + V(afterstate): {"action", "state", "reward", "value"} (``ops.ntuple_greedy``)."""
        return ops.ntuple_greedy(board, self.weights, self.tuples, reward_fn=reward_fn, action_dtype=action_dtype, out=out,
                                 stages=self.stages, promoted=self.promoted)

    def expectimax(self, board: torch.Tensor, *, depth: int = 1, two_prob: float = 0.8, reward_fn=None,
                   action_dtype: torch.dtype = torch.int64, out: Optional[dict] = None) -> dict:
        """The expectimax move ``depth`` (1 or 2) chance layers deep: {"action", "state", "reward", "value", "q"}
        (``ops.ntuple_expectimax``)."""
        return ops.ntuple_expectimax(board, self.weights, self.tuples, depth=depth, two_prob=two_prob, reward_fn=reward_fn,
                                     action_dtype=action_dtype, out=out, stages=self.stages, promoted=self.promoted)

    def td_update(self, afterstate: torch.Tensor, target: torch.Tensor, alpha: float, *, mask: Optional[torch.Tensor] = None,
                  delta_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One synchronous TD(0) batch toward ``target``; returns delta = alpha * (target - V) (``ops.ntuple_td_update``).
        The adds are float atomics: the weights are reproducible up to the fp32 rounding of their order."""
        return ops.ntuple_td_update(afterstate, target, self.weights, self.tuples, alpha=alpha, mask=mask, delta_out=delta_out,
                                    stages=self.stages, promoted=self.promoted)

    def _tc_alloc(self) -> None:
        if self.coherence is None:
            self.coherence = torch.zeros((self.weights.numel(), 2), dtype=torch.float32, device=self.device)
        if self._tc_accum is None:
            self._tc_accum = torch.zeros((self.weights.numel(), 2), dtype=torch.float32, device=self.device)

    def tc_update(self, afterstate: torch.Tensor, target: torch.Tensor, alpha: float, *, mask: Optional[torch.Tensor] = None,
                  delta_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One synchronous temporal coherence batch toward ``target``; returns delta = alpha * (target - V)
        (``ops.ntuple_tc_update``).  The first call allocates ``coherence`` ((S * N, 2) float32 {E, A} per weight, zeros)
        and a zero scratch accumulator of the same shape."""
        self._tc_alloc()
        return ops.ntuple_tc_update(afterstate, target, self.weights, self.coherence, self._tc_accum, self.tuples, alpha=alpha,
                                    mask=mask, delta_out=delta_out, stages=self.stages, promoted=self.promoted)

    def td_lambda_update(self, after_ring: torch.Tensor, reward_ring: torch.Tensor, ended_ring: torch.Tensor, newest: int,
                         alpha: float, lam: float, *, mask: Optional[torch.Tensor] = None,
                         delta_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One synchronous delayed TD(lambda) batch over the caller's ring of each game's last h + 1 afterstates; returns
        delta = alpha * (R_0 - V(x_0)) (``ops.ntuple_td_lambda_update``)."""
        return ops.ntuple_td_lambda_update(after_ring, reward_ring, ended_ring, newest, self.weights, self.tuples, alpha=alpha,
                                           lam=lam, mask=mask, delta_out=delta_out, stages=self.stages, promoted=self.promoted)

    def tc_lambda_update(self, after_ring: torch.Tensor, reward_ring: torch.Tensor, ended_ring: torch.Tensor, newest: int,
                         alpha: float, lam: float, *, mask: Optional[torch.Tensor] = None,
                         delta_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One synchronous delayed TC(lambda) batch (``ops.ntuple_tc_lambda_update``); ``coherence`` and the scratch
        accumulator are allocated as by ``tc_update``."""
        self._tc_alloc()
        return ops.ntuple_tc_lambda_update(after_ring, reward_ring, ended_ring, newest, self.weights, self.coherence,
                                           self._tc_accum, self.tuples, alpha=alpha, lam=lam, mask=mask, delta_out=delta_out,
                                           stages=self.stages, promoted=self.promoted)

    def state_dict(self) -> dict:
        state = {"tuples": [list(t) for t in self.tuples], "stages": list(self.stages), "weights": self.weights.detach().clone()}
        if self.coherence is not None:
            state["coherence"] = self.coherence.detach().clone()
        if self.promoted is not None:
            state["promoted"] = self.promoted.detach().clone()
        return state

    def load_state_dict(self, state: dict) -> None:
        """Loads the weights and, when ``state`` has them, the TC coherence sums; a dict without ``"coherence"`` drops any
        coherence state this network has (the next ``tc_update`` starts from zeros).  A dict without ``"stages"`` is a
        single-stage network's (``stages=()``).

        Promotion marks (``"promoted"``): a promoting network copies them from a dict that has them; from a dict without them
        it sets every stage's mark (bits 0..S-2) of every entry, so that it values every board as the saved network did.  A
        non-promoting network loads a dict with marks as its effective weights (``ops.ntuple_promoted_weights``), with the
        coherence of every unmarked entry of stages >= 1 zeroed, as a promotion would set it."""
        if ops.ntuple_spec(state["tuples"]) != self.tuples:
            raise ValueError(f"state_dict is for tuples {state['tuples']}, this network has {self.tuples}")
        if ops.ntuple_stages(state.get("stages", ())) != self.stages:
            raise ValueError(f"state_dict is for stages {tuple(state.get('stages', ()))}, this network has {self.stages}")
        w = state["weights"]
        if not isinstance(w, torch.Tensor) or w.dtype != torch.float32 or tuple(w.shape) != tuple(self.weights.shape):
            raise ValueError(f"weights must be float32 {tuple(self.weights.shape)}")
        c = state.get("coherence")
        shape = (self.weights.numel(), 2)
        if c is not None and (not isinstance(c, torch.Tensor) or c.dtype != torch.float32 or tuple(c.shape) != shape):
            raise ValueError(f"coherence must be float32 {shape}")
        p = state.get("promoted")
        n = self.weights.numel() // (len(self.stages) + 1)
        if p is not None and (not isinstance(p, torch.Tensor) or p.dtype != torch.uint8 or tuple(p.shape) != (n,)):
            raise ValueError(f"promoted must be uint8 ({n},)")
        if p is not None and self.promoted is None:
            # marks into a network without them: the effective weights, and the coherence a promotion would leave
            p = p.detach().to(self.device).contiguous()
            w = ops.ntuple_promoted_weights(w.detach().to(self.device).contiguous(), p, self.tuples, self.stages)
            if c is not None:
                c = c.detach().to(self.device, copy=True).contiguous()
                marked = torch.ones((len(self.stages) + 1, n), dtype=torch.bool, device=self.device)
                for s in range(1, len(self.stages) + 1):
                    marked[s] = (p & (1 << (s - 1))) != 0
                c[~marked.view(-1)] = 0.0
        self.weights.copy_(w)
        if self.promoted is not None:
            if p is None:
                self.promoted.fill_((1 << len(self.stages)) - 1)
            else:
                self.promoted.copy_(p)
        if c is None:
            self.coherence = None
        elif self.coherence is None:
            self.coherence = c.detach().to(self.device, copy=True).contiguous()
        else:
            self.coherence.copy_(c)


class GreedyPolicy:
    """The network's greedy afterstate move as a policy ``DeviceRunner`` accepts: ``sample_actions(state, valid_actions)``
    returns (actions int64, log_probs 0).  ``reward_fn`` must be the environment's.  A multi-stage network works here as is."""

    def __init__(self, net: NTupleNetwork, reward_fn=None):
        self.net = net
        self.reward_fn = reward_fn

    def sample_actions(self, state: torch.Tensor, valid_actions: torch.Tensor):
        board = state.to(self.net.device, torch.uint8).contiguous()  # exponents fit a byte
        actions = self.net.greedy(board, reward_fn=self.reward_fn)["action"]
        return actions, torch.zeros(actions.shape, dtype=torch.float32, device=actions.device)


class ExpectimaxPolicy:
    """The network's expectimax move (``NTupleNetwork.expectimax``) as a policy ``DeviceRunner`` accepts:
    ``sample_actions(state, valid_actions)`` returns (actions int64, log_probs 0).  ``reward_fn`` and ``two_prob`` must be the
    environment's: the search scores moves with that reward and averages over spawns with that chance of a 2.  A multi-stage
    network works here as is: each leaf is valued with its own stage's tables."""

    def __init__(self, net: NTupleNetwork, depth: int = 1, reward_fn=None, two_prob: float = 0.8):
        if isinstance(depth, bool) or depth not in (1, 2):
            raise ValueError(f"depth must be 1 or 2, got {depth!r}")
        self.net = net
        self.depth = depth
        self.reward_fn = reward_fn
        self.two_prob = two_prob

    def sample_actions(self, state: torch.Tensor, valid_actions: torch.Tensor):
        board = state.to(self.net.device, torch.uint8).contiguous()  # exponents fit a byte
        actions = self.net.expectimax(board, depth=self.depth, two_prob=self.two_prob, reward_fn=self.reward_fn)["action"]
        return actions, torch.zeros(actions.shape, dtype=torch.float32, device=actions.device)


class TDAfterstateLearner:
    """TD(0) afterstate learning over a device-resident ``VecGame(..., output="torch", sync_free=True)``.

    ``step()`` runs one iteration for all M games without a host synchronisation:

    1. ``env.prepare()`` (games that ended in the previous step restart);
    2. greedy afterstate move on the boards (``NTupleNetwork.greedy``);
    3. TD(0) (or, with ``rule="tc"``, TC) update of each game's previous afterstate toward reward + value of the move just
       chosen, or toward 0 for a game that ended in the previous step; games without a previous afterstate (the first step
       after ``reset()``) are masked out;
    4. ``env.step(action)``.

    ``alpha`` defaults to ``default_alpha(M)``.  With ``alpha=0`` step 3 is skipped and the learner plays the greedy policy
    (evaluation).  Call ``reset(seed)`` instead of ``env.reset`` so that no afterstate of the old games is updated.

    ``rule``: ``"td0"`` (the default) updates with ``NTupleNetwork.td_update``; ``"tc"`` with temporal coherence learning
    (``NTupleNetwork.tc_update``: a step size per weight), whose ``alpha`` defaults to ``default_tc_alpha(M)``.

    ``horizon`` = h > 1 makes the rule delayed TD(lambda) / TC(lambda) (``NTupleNetwork.td_lambda_update`` /
    ``tc_lambda_update``, lambda = ``lam``): the learner keeps each game's last h + 1 afterstates, rewards and end flags in a
    ring, and step T (counted from ``reset()``) writes x_T and its reward into slot T mod (h + 1) straight from the greedy
    kernel and, after ``env.step``, the game's end flag.  Steps 0 .. h-1 update nothing; from step h on, each step updates
    the afterstate of step T - h (slot (T + 1) mod (h + 1)) toward the lambda-return over the window up to x_T, truncated at
    the first end in it.  So the last h afterstates of a run are never updated.  ``delta`` is the delta of the afterstate
    updated in the step (0 while nothing is).  With ``rule="tc"`` and h > 1, ``alpha`` defaults to
    ``DEFAULT_TC_LAMBDA_ALPHA_TIMES_GAMES / M``.  ``horizon=1`` is the TD(0) / TC learner above, whatever ``lam`` is.

    A multi-stage network (``NTupleNetwork(..., stages=...)``) works with every rule: the learner only calls the network.
    The default step sizes are the single-stage sweeps'; none has been run for staged networks."""

    def __init__(self, env, net: NTupleNetwork, alpha: Optional[float] = None, rule: str = "td0", horizon: int = 1,
                 lam: float = 0.5):
        if env._output != "torch" or not env._sync_free:
            raise ValueError("TDAfterstateLearner needs VecGame(..., output='torch', sync_free=True)")
        if env.device != net.device:
            raise ValueError(f"the environment is on {env.device}, the network on {net.device}")
        if rule not in ("td0", "tc"):
            raise ValueError(f"rule must be 'td0' or 'tc', got {rule!r}")
        if isinstance(horizon, bool) or not isinstance(horizon, int) or not 1 <= horizon <= ops.NTUPLE_LAMBDA_MAX_HORIZON:
            raise ValueError(f"horizon must be an int in 1..{ops.NTUPLE_LAMBDA_MAX_HORIZON}, got {horizon!r}")
        if isinstance(lam, bool) or not isinstance(lam, (int, float)) or not 0.0 <= lam <= 1.0:
            raise ValueError(f"lam must be a number in [0, 1], got {lam!r}")
        self.horizon, self.lam = horizon, float(lam)
        self.env, self.net, self.rule = env, net, rule
        if alpha is not None:
            self.alpha = float(alpha)
        else:
            self.alpha = default_tc_alpha(env._size) if rule == "tc" else default_alpha(env._size)
            if rule == "tc" and horizon > 1:
                self.alpha = DEFAULT_TC_LAMBDA_ALPHA_TIMES_GAMES / env._size
        self._update = net.tc_update if rule == "tc" else net.td_update
        m, dev = env._size, env.device
        self._out = {"action": torch.zeros((m,), dtype=torch.uint8, device=dev),
                     "state": torch.zeros((m, 16), dtype=torch.uint8, device=dev),
                     "reward": torch.zeros((m,), dtype=torch.float32, device=dev),
                     "value": torch.zeros((m,), dtype=torch.float32, device=dev)}
        self._prev_after = torch.zeros((m, 16), dtype=torch.uint8, device=dev)
        self._prev_ended = torch.zeros((m,), dtype=torch.bool, device=dev)  # prepare() clears env's terminated: our own copy
        self._has_prev = torch.zeros((m,), dtype=torch.uint8, device=dev)
        self._target = torch.zeros((m,), dtype=torch.float32, device=dev)
        self.delta = torch.zeros((m,), dtype=torch.float32, device=dev)  # the last update's alpha * TD error (0: masked out)
        if horizon > 1:
            slots = horizon + 1
            self._lambda_update = net.tc_lambda_update if rule == "tc" else net.td_lambda_update
            self._after_ring = torch.zeros((slots, m, 16), dtype=torch.uint8, device=dev)
            self._reward_ring = torch.zeros((slots, m), dtype=torch.float32, device=dev)
            self._ended_ring = torch.zeros((slots, m), dtype=torch.uint8, device=dev)
            self._ring_out = [dict(self._out, state=self._after_ring[s], reward=self._reward_ring[s]) for s in range(slots)]
            self._steps = 0  # steps since reset(): the window is full from step h on

    def reset(self, seed: Optional[int] = None) -> None:
        self.env.reset(seed)
        self._has_prev.zero_()
        if self.horizon > 1:
            self._steps = 0
            self.delta.zero_()

    def step(self):
        if self.horizon > 1:
            return self._step_lambda()
        env = self.env
        env.prepare()
        board = env.observations()[0]
        g = self.net.greedy(board, reward_fn=env._reward_fn, action_dtype=torch.uint8, out=self._out)
        if self.alpha != 0.0:
            torch.add(g["reward"], g["value"], out=self._target)
            self._target.masked_fill_(self._prev_ended, 0.0)
            self._update(self._prev_after, self._target, self.alpha, mask=self._has_prev, delta_out=self.delta)
        res = env.step(g["action"])
        self._prev_after.copy_(g["state"])
        self._prev_ended.copy_(res["terminated"])
        self._has_prev.fill_(1)
        return res

    def _step_lambda(self):
        env, h = self.env, self.horizon
        env.prepare()
        board = env.observations()[0]
        newest = self._steps % (h + 1)
        g = self.net.greedy(board, reward_fn=env._reward_fn, action_dtype=torch.uint8, out=self._ring_out[newest])
        if self.alpha != 0.0 and self._steps >= h:
            self._lambda_update(self._after_ring, self._reward_ring, self._ended_ring, newest, self.alpha, self.lam,
                                delta_out=self.delta)
        res = env.step(g["action"])
        self._ended_ring[newest].copy_(res["terminated"])
        self._steps += 1
        return res
