"""N-tuple value networks on the device and a TD(0) afterstate learner over ``VecGame``.

An n-tuple network (Szubert & Jaskowski 2014; Yeh et al. 2016) values a 2048 board as a sum of table entries indexed by the
4-bit fields of a few cells, over the board's 8 symmetric images (one table per tuple, shared by the images).  Evaluating it,
choosing the greedy afterstate move with it and updating it are integer byte work on boards plus scattered 4-byte reads and
adds: each is one kernel here (``ops.ntuple_value``, ``ops.ntuple_greedy``, ``ops.ntuple_td_update``).

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
# 0.8 / 1.6 / 3.2 at all three sizes), and c = 0.4 is the best of them.
DEFAULT_ALPHA_TIMES_GAMES = 0.4


def default_alpha(num_games: int) -> float:
    return DEFAULT_ALPHA_TIMES_GAMES / num_games


class NTupleNetwork:
    """An n-tuple value function with its weights on one CUDA device.

    ``tuples``: 1..16 tuples of 1..6 distinct cells (cell = row*4 + col).  The weights are one zero-initialised float32 tensor
    of sum 16^len entries, tuple t's table after those of the tuples before it (``offsets``)."""

    def __init__(self, tuples=STANDARD_4X6, device: Any = None):
        self.tuples = ops.ntuple_spec(tuples)
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
        self.weights = torch.zeros((total,), dtype=torch.float32, device=dev)

    def value(self, board: torch.Tensor, *, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """V of (M,16) boards: (M,) float32 (``ops.ntuple_value``)."""
        return ops.ntuple_value(board, self.weights, self.tuples, out=out)

    def greedy(self, board: torch.Tensor, *, reward_fn=None, action_dtype: torch.dtype = torch.int64,
               out: Optional[dict] = None) -> dict:
        """The move maximising reward + V(afterstate): {"action", "state", "reward", "value"} (``ops.ntuple_greedy``)."""
        return ops.ntuple_greedy(board, self.weights, self.tuples, reward_fn=reward_fn, action_dtype=action_dtype, out=out)

    def td_update(self, afterstate: torch.Tensor, target: torch.Tensor, alpha: float, *, mask: Optional[torch.Tensor] = None,
                  delta_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One synchronous TD(0) batch toward ``target``; returns delta = alpha * (target - V) (``ops.ntuple_td_update``).
        The adds are float atomics: the weights are reproducible up to the fp32 rounding of their order."""
        return ops.ntuple_td_update(afterstate, target, self.weights, self.tuples, alpha=alpha, mask=mask, delta_out=delta_out)

    def state_dict(self) -> dict:
        return {"tuples": [list(t) for t in self.tuples], "weights": self.weights.detach().clone()}

    def load_state_dict(self, state: dict) -> None:
        if ops.ntuple_spec(state["tuples"]) != self.tuples:
            raise ValueError(f"state_dict is for tuples {state['tuples']}, this network has {self.tuples}")
        w = state["weights"]
        if not isinstance(w, torch.Tensor) or w.dtype != torch.float32 or tuple(w.shape) != tuple(self.weights.shape):
            raise ValueError(f"weights must be float32 {tuple(self.weights.shape)}")
        self.weights.copy_(w)


class GreedyPolicy:
    """The network's greedy afterstate move as a policy ``DeviceRunner`` accepts: ``sample_actions(state, valid_actions)``
    returns (actions int64, log_probs 0).  ``reward_fn`` must be the environment's."""

    def __init__(self, net: NTupleNetwork, reward_fn=None):
        self.net = net
        self.reward_fn = reward_fn

    def sample_actions(self, state: torch.Tensor, valid_actions: torch.Tensor):
        board = state.to(self.net.device, torch.uint8).contiguous()  # exponents fit a byte
        actions = self.net.greedy(board, reward_fn=self.reward_fn)["action"]
        return actions, torch.zeros(actions.shape, dtype=torch.float32, device=actions.device)


class TDAfterstateLearner:
    """TD(0) afterstate learning over a device-resident ``VecGame(..., output="torch", sync_free=True)``.

    ``step()`` runs one iteration for all M games without a host synchronisation:

    1. ``env.prepare()`` (games that ended in the previous step restart);
    2. greedy afterstate move on the boards (``NTupleNetwork.greedy``);
    3. TD(0) update of each game's previous afterstate toward reward + value of the move just chosen, or toward 0 for a
       game that ended in the previous step; games without a previous afterstate (the first step after ``reset()``) are
       masked out;
    4. ``env.step(action)``.

    ``alpha`` defaults to ``default_alpha(M)``.  With ``alpha=0`` step 3 is skipped and the learner plays the greedy policy
    (evaluation).  Call ``reset(seed)`` instead of ``env.reset`` so that no afterstate of the old games is updated."""

    def __init__(self, env, net: NTupleNetwork, alpha: Optional[float] = None):
        if env._output != "torch" or not env._sync_free:
            raise ValueError("TDAfterstateLearner needs VecGame(..., output='torch', sync_free=True)")
        if env.device != net.device:
            raise ValueError(f"the environment is on {env.device}, the network on {net.device}")
        self.env, self.net = env, net
        self.alpha = default_alpha(env._size) if alpha is None else float(alpha)
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

    def reset(self, seed: Optional[int] = None) -> None:
        self.env.reset(seed)
        self._has_prev.zero_()

    def step(self):
        env = self.env
        env.prepare()
        board = env.observations()[0]
        g = self.net.greedy(board, reward_fn=env._reward_fn, action_dtype=torch.uint8, out=self._out)
        if self.alpha != 0.0:
            torch.add(g["reward"], g["value"], out=self._target)
            self._target.masked_fill_(self._prev_ended, 0.0)
            self.net.td_update(self._prev_after, self._target, self.alpha, mask=self._has_prev, delta_out=self.delta)
        res = env.step(g["action"])
        self._prev_after.copy_(g["state"])
        self._prev_ended.copy_(res["terminated"])
        self._has_prev.fill_(1)
        return res
