"""Stand-alone device ops of the rollout path (thin wrappers over the C ABI, torch CUDA tensors in and out).

    sample_masked_categorical   _sample_action, policy/actor_critic.py:56-76
    gae_advantages              the recurrence of compute_gae, gae.py:50, :65-68
    encode_onehot               CNNEncoder.forward's input encoding, policy/_network.py:86-95
    valid_actions               _compute_valid_actions, game_numba.py:259-289
    afterstates                 all four moves of every board up to the spawn: _step_kernel + reward_fn, game_numba.py:93-134,
                                :408-504 at :728 (moved board, reward, "the move changes the board", optionally `merged`)
    ntuple_value, ntuple_greedy, ntuple_td_update
                                an n-tuple network's value, greedy afterstate move and TD(0) batch update (no reference
                                counterpart; ml2048_b200.ntuple wraps them)
"""

from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import _lib
from .rewards import reward_kind

_ONEHOT = {torch.float32: _lib.ONEHOT_F32, torch.bfloat16: _lib.ONEHOT_BF16, torch.uint8: _lib.ONEHOT_U8}


def _stream(t: torch.Tensor) -> int:
    from .vecgame import _raw_stream

    return _raw_stream(t.device.index)


def _cuda(t: torch.Tensor, name: str) -> None:
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous()):
        raise ValueError(f"{name} must be a contiguous CUDA tensor")


def sample_masked_categorical(logits: torch.Tensor, valid: torch.Tensor, *, seed: int, counter: int, slot_base: int = 0,
                              dtype: torch.dtype = torch.int64) -> tuple[torch.Tensor, torch.Tensor]:
    """Sample one action per game from softmax(logits restricted to valid) and return (actions, log_probs).

    Same distribution and log-probabilities as the reference's ``_sample_action`` (invalid actions masked to
    finfo.min, ``Categorical(logits=...)``); the uniform comes from Philox2x32-10 keyed by
    (seed, slot_base + game, counter) -- the policy word the step kernel itself draws -- instead of ``torch.multinomial``'s generator."""
    _cuda(logits, "logits")
    _cuda(valid, "valid")
    if logits.dtype != torch.float32 or logits.ndim != 2 or logits.shape[1] != 4:
        raise ValueError(f"logits must be float32 (M,4), got {logits.dtype}{tuple(logits.shape)}")
    if valid.shape != logits.shape or valid.dtype not in (torch.bool, torch.uint8):
        raise ValueError(f"valid must be bool/uint8 {tuple(logits.shape)}")
    if dtype not in (torch.int64, torch.uint8):
        raise ValueError("dtype must be torch.int64 or torch.uint8")
    m = logits.shape[0]
    actions = torch.empty((m,), dtype=dtype, device=logits.device)
    log_prob = torch.empty((m,), dtype=torch.float32, device=logits.device)
    lib = _lib.load()
    with torch.cuda.device(logits.device):
        rc = lib.ml2048_sample_masked_categorical(
            logits.data_ptr(), valid.data_ptr(), actions.data_ptr() if dtype == torch.uint8 else None,
            actions.data_ptr() if dtype == torch.int64 else None, log_prob.data_ptr(), m, int(slot_base),
            int(seed) & 0xFFFFFFFFFFFFFFFF, int(counter) & 0xFFFFFFFFFFFFFFFF, _stream(logits))
    _lib.check(rc, "ml2048_sample_masked_categorical")
    return actions, log_prob


def gae_advantages(v0: torch.Tensor, v1: torch.Tensor, reward: torch.Tensor, terminated: torch.Tensor, *, gamma: float,
                   lambda_: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Generalised advantage estimation over (use, step, game) tensors, as ``compute_gae`` (gae.py:50, :65-68):
    ``delta = gamma*v1*~terminated + reward - v0`` then the reverse scan with ``coef = gamma*lambda_``.
    One kernel instead of 3 torch ops per step; same fp32 rounding as the reference's ops."""
    for name, t in (("v0", v0), ("v1", v1), ("reward", reward), ("terminated", terminated)):
        _cuda(t, name)
    if v0.ndim != 3 or v0.dtype != torch.float32:
        raise ValueError(f"v0 must be float32 (use, step, game), got {v0.dtype}{tuple(v0.shape)}")
    if v1.shape != v0.shape or reward.shape != v0.shape or terminated.shape != v0.shape:
        raise ValueError("v0, v1, reward, terminated must have the same shape")
    if v1.dtype != torch.float32 or reward.dtype != torch.float32 or terminated.dtype not in (torch.bool, torch.uint8):
        raise ValueError("v1/reward must be float32 and terminated bool/uint8")
    if out is None:
        out = torch.empty_like(v0)
    _cuda(out, "out")
    if out.shape != v0.shape or out.dtype != torch.float32:
        raise ValueError("out must be float32 with the shape of v0")
    u, s, g = v0.shape
    lib = _lib.load()
    with torch.cuda.device(v0.device):
        rc = lib.ml2048_gae(v0.data_ptr(), v1.data_ptr(), reward.data_ptr(), terminated.data_ptr(), out.data_ptr(), u, s, g,
                            float(gamma), float(gamma * lambda_), _stream(v0))
    _lib.check(rc, "ml2048_gae")
    return out


def encode_onehot(board: torch.Tensor, dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """(M,16) uint8 boards -> (M,16,16) class-major one-hot == F.one_hot(x,16).to(dtype).permute(0,2,1)."""
    _cuda(board, "board")
    if board.dtype not in (torch.uint8, torch.int8) or board.ndim != 2 or board.shape[1] != 16:
        raise ValueError("board must be uint8/int8 (M,16)")
    if dtype not in _ONEHOT:
        raise ValueError(f"dtype {dtype} not supported")
    out = torch.empty((board.shape[0], 16, 16), dtype=dtype, device=board.device)
    lib = _lib.load()
    with torch.cuda.device(board.device):
        rc = lib.ml2048_encode_onehot(board.data_ptr(), out.data_ptr(), _ONEHOT[dtype], board.shape[0], _stream(board))
    _lib.check(rc, "ml2048_encode_onehot")
    return out


def valid_actions(board: torch.Tensor) -> torch.Tensor:
    """(M,16) uint8 boards -> (M,4) uint8 masks (left, right, up, down)."""
    _cuda(board, "board")
    if board.dtype not in (torch.uint8, torch.int8) or board.ndim != 2 or board.shape[1] != 16:
        raise ValueError("board must be uint8/int8 (M,16)")
    out = torch.empty((board.shape[0], 4), dtype=torch.uint8, device=board.device)
    lib = _lib.load()
    with torch.cuda.device(board.device):
        rc = lib.ml2048_valid_actions(board.data_ptr(), out.data_ptr(), board.shape[0], _stream(board))
    _lib.check(rc, "ml2048_valid_actions")
    return out


# afterstates() outputs: key (VecStepResult's names) -> (shape after M, dtype)
_AFTERSTATES = {
    "state": ((4, 16), torch.uint8),
    "reward": ((4,), torch.float32),
    "valid_actions": ((4,), torch.uint8),
    "merged": ((4, 16), torch.uint8),
}


def afterstates(board: torch.Tensor, *, reward_fn=None, merged: bool = False, out: Optional[dict] = None) -> dict:
    """The four moves of every board, without the spawn and without touching any environment state.

    ``board``: (M,16) uint8/int8 boards.  Returns a dict of CUDA tensors, direction-major per board (0 left, 1 right,
    2 up, 3 down):

        "state"          (M,4,16) uint8    the board after the move (no tile spawned)
        "reward"         (M,4)    float32  reward_fn of that move, bit for bit what step(a) returns; 0 where the move
                                           does not change the board
        "valid_actions"  (M,4)    uint8    1 iff the move changes the board (== ops.valid_actions(board))
        "merged"         (M,4,16) uint8    only with merged=True: fusions per exponent, as step() logs them

    ``reward_fn`` selects one of the four reward functions like ``VecGame(reward_fn=...)`` (default: normal).
    ``out``: preallocated tensors under the same keys (any subset; "merged" only with merged=True), so that the call can be
    captured in a CUDA graph.  Cells must be 0..17, as for every op here; nothing is checked on the device."""
    if not isinstance(board, torch.Tensor) or board.dtype not in (torch.uint8, torch.int8) or board.ndim != 2 or board.shape[1] != 16:
        raise ValueError("board must be uint8/int8 (M,16)")
    kind = reward_kind(reward_fn)
    keys = ("state", "reward", "valid_actions", "merged") if merged else ("state", "reward", "valid_actions")
    out = {} if out is None else out
    if not isinstance(out, dict):
        raise ValueError("out must be a dict of tensors")
    unknown = set(out) - set(keys)
    if unknown:
        raise ValueError(f"out has entries afterstates does not write: {sorted(unknown)}")
    _cuda(board, "board")
    m = board.shape[0]
    res = {}
    for k in keys:
        shape, dtype = _AFTERSTATES[k]
        shape = (m,) + shape
        t = out.get(k)
        if t is None:
            t = torch.empty(shape, dtype=dtype, device=board.device)
        elif not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous() and t.dtype == dtype and tuple(t.shape) == shape
                  and t.device == board.device):
            raise ValueError(f"out[{k!r}] must be a contiguous {dtype} tensor {shape} on {board.device}")
        res[k] = t
    if m == 0:
        return res
    lib = _lib.load()
    with torch.cuda.device(board.device):
        rc = lib.ml2048_afterstates(board.data_ptr(), res["state"].data_ptr(), res["reward"].data_ptr(), res["valid_actions"].data_ptr(),
                                    res["merged"].data_ptr() if merged else None, kind, m, _stream(board))
    _lib.check(rc, "ml2048_afterstates")
    return res


# ---- n-tuple networks ----------------------------------------------------------------------------------------------------

NTUPLE_MAX_TUPLES, NTUPLE_MAX_LEN = 16, 6


def ntuple_spec(tuples) -> tuple:
    """Check an n-tuple network's tuples on the host and return them as a tuple of tuples of ints.

    1 to 16 tuples, each 1 to 6 distinct cells in 0..15 (cell = row*4 + col).  Raises ValueError otherwise."""
    try:
        spec = tuple(tuple(int(c) for c in t) for t in tuples)
    except TypeError:
        raise ValueError("tuples must be a sequence of sequences of cells") from None
    if not 1 <= len(spec) <= NTUPLE_MAX_TUPLES:
        raise ValueError(f"an n-tuple network has 1..{NTUPLE_MAX_TUPLES} tuples, got {len(spec)}")
    for t in spec:
        if not 1 <= len(t) <= NTUPLE_MAX_LEN:
            raise ValueError(f"a tuple has 1..{NTUPLE_MAX_LEN} cells, got {t}")
        if any(c < 0 or c > 15 for c in t) or len(set(t)) != len(t):
            raise ValueError(f"a tuple's cells are distinct and in 0..15, got {t}")
    return spec


def ntuple_num_weights(tuples) -> int:
    """sum over the tuples of 16^len: the length of the network's one float32 weight tensor"""
    return sum(16 ** len(t) for t in ntuple_spec(tuples))


_SPEC_ARRAYS: dict = {}


def _spec_arrays(tuples):
    """(cells [K][6] u8, len [K] u8, K, number of weights) of checked tuples, cached per spec"""
    key = tuples if isinstance(tuples, tuple) else None
    got = _SPEC_ARRAYS.get(key) if key is not None else None
    if got is None:
        spec = ntuple_spec(tuples)
        cells = np.zeros((len(spec), NTUPLE_MAX_LEN), np.uint8)
        for i, t in enumerate(spec):
            cells[i, :len(t)] = t
        got = (cells, np.array([len(t) for t in spec], np.uint8), len(spec), sum(16 ** len(t) for t in spec))
        if key is not None and len(_SPEC_ARRAYS) < 64:
            _SPEC_ARRAYS[key] = got
    return got


def _weights_arg(weights: torch.Tensor, n: int, device) -> None:
    if not (isinstance(weights, torch.Tensor) and weights.is_cuda and weights.is_contiguous() and weights.dtype == torch.float32
            and weights.ndim == 1):
        raise ValueError("weights must be a contiguous 1-D float32 CUDA tensor")
    if weights.numel() != n:
        raise ValueError(f"weights has {weights.numel()} entries, the tuples need sum 16^len = {n}")
    if weights.device != device:
        raise ValueError(f"weights is on {weights.device}, the boards on {device}")


def _board_arg(board, name: str = "board") -> None:
    if not isinstance(board, torch.Tensor) or board.dtype not in (torch.uint8, torch.int8) or board.ndim != 2 or board.shape[1] != 16:
        raise ValueError(f"{name} must be uint8/int8 (M,16)")
    _cuda(board, name)


def _out_arg(t, shape: tuple, dtype, device, name: str) -> torch.Tensor:
    if t is None:
        return torch.empty(shape, dtype=dtype, device=device)
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous() and t.dtype == dtype and tuple(t.shape) == shape
            and t.device == device):
        raise ValueError(f"{name} must be a contiguous {dtype} tensor {shape} on {device}")
    return t


def ntuple_value(board: torch.Tensor, weights: torch.Tensor, tuples, *, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """V(board) of an n-tuple network: (M,16) uint8/int8 boards -> (M,) float32.

    ``tuples``: the network's cells (see ``ntuple_spec``); ``weights``: its one float32 tensor of sum 16^len entries, tuple t's
    table after those of tuples 0..t-1.  V sums, for t = 0..K-1 and then each of the board's 8 symmetric images g = 0..7,
    ``weights[offset_t + sum_j min(image_g[cell_tj], 15) << 4j]`` as float32 adds from 0 in that order: bit-reproducible.
    Every byte gives an in-bounds index; tiles 2^16 and above share the entries of 2^15.  ``out``: a preallocated (M,)
    float32 tensor (CUDA-graph capture)."""
    _board_arg(board)
    cells, lens, k, n = _spec_arrays(tuples)
    _weights_arg(weights, n, board.device)
    m = board.shape[0]
    out = _out_arg(out, (m,), torch.float32, board.device, "out")
    if m == 0:
        return out
    lib = _lib.load()
    with torch.cuda.device(board.device):
        rc = lib.ml2048_ntuple_value(board.data_ptr(), weights.data_ptr(), n, cells.ctypes.data, lens.ctypes.data, k, out.data_ptr(), m,
                                     _stream(board))
    _lib.check(rc, "ml2048_ntuple_value")
    return out


_NTUPLE_GREEDY = {"state": ((16,), torch.uint8), "reward": ((), torch.float32), "value": ((), torch.float32)}


def ntuple_greedy(board: torch.Tensor, weights: torch.Tensor, tuples, *, reward_fn=None, action_dtype: torch.dtype = torch.int64,
                  out: Optional[dict] = None) -> dict:
    """The greedy afterstate move of every board under an n-tuple network, in one kernel.

    For every direction a that changes the board, q_a = reward_a + V(afterstate_a) in float32, with reward_a and afterstate_a
    exactly ``afterstates(board, reward_fn=reward_fn)``'s.  The largest q wins; NaN ranks as -inf; ties go to the smallest a.
    Returns a dict of CUDA tensors:

        "action"  (M,)    action_dtype (int64 or uint8)
        "state"   (M,16)  uint8    the chosen afterstate (no tile spawned)
        "reward"  (M,)    float32  its reward
        "value"   (M,)    float32  V(afterstate)

    A board without a valid move gets action 0, its own board, reward 0 and value 0 (so a TD target reward + value is 0).
    ``out``: preallocated tensors under the same keys (any subset), so that the call can be captured in a CUDA graph."""
    _board_arg(board)
    if action_dtype not in (torch.int64, torch.uint8):
        raise ValueError("action_dtype must be torch.int64 or torch.uint8")
    kind = reward_kind(reward_fn)
    cells, lens, k, n = _spec_arrays(tuples)
    _weights_arg(weights, n, board.device)
    out = {} if out is None else out
    if not isinstance(out, dict):
        raise ValueError("out must be a dict of tensors")
    unknown = set(out) - {"action", *_NTUPLE_GREEDY}
    if unknown:
        raise ValueError(f"out has entries ntuple_greedy does not write: {sorted(unknown)}")
    m = board.shape[0]
    res = {"action": _out_arg(out.get("action"), (m,), action_dtype, board.device, "out['action']")}
    for key, (shape, dtype) in _NTUPLE_GREEDY.items():
        res[key] = _out_arg(out.get(key), (m,) + shape, dtype, board.device, f"out[{key!r}]")
    if m == 0:
        return res
    act = res["action"].data_ptr()
    lib = _lib.load()
    with torch.cuda.device(board.device):
        rc = lib.ml2048_ntuple_greedy(board.data_ptr(), weights.data_ptr(), n, cells.ctypes.data, lens.ctypes.data, k, kind,
                                      act if action_dtype == torch.uint8 else None, act if action_dtype == torch.int64 else None,
                                      res["state"].data_ptr(), res["reward"].data_ptr(), res["value"].data_ptr(), m, _stream(board))
    _lib.check(rc, "ml2048_ntuple_greedy")
    return res


def ntuple_td_update(afterstate: torch.Tensor, target: torch.Tensor, weights: torch.Tensor, tuples, *, alpha: float,
                     mask: Optional[torch.Tensor] = None, delta_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One synchronous batch of TD(0) updates of an n-tuple network, in place on ``weights``; returns delta (M,) float32.

    Phase 1: delta_i = alpha * (target_i - V(afterstate_i)) with the weights as they were before the call, 0 for a game
    whose ``mask`` byte is 0 (``mask``: (M,) bool/uint8, None = every game).  Phase 2: every entry of every masked-in game,
    8 per tuple, gets += delta_i.  Phase 2 adds with float atomics, so the order of the adds that several games make to one
    entry is unspecified: the weights are reproducible only up to the fp32 rounding of that order.  delta is deterministic.
    ``delta_out``: a preallocated (M,) float32 tensor (CUDA-graph capture)."""
    _board_arg(afterstate, "afterstate")
    m = afterstate.shape[0]
    _cuda(target, "target")
    if target.dtype != torch.float32 or tuple(target.shape) != (m,):
        raise ValueError(f"target must be float32 ({m},)")
    if mask is not None:
        _cuda(mask, "mask")
        if mask.dtype not in (torch.bool, torch.uint8) or tuple(mask.shape) != (m,):
            raise ValueError(f"mask must be bool/uint8 ({m},)")
    cells, lens, k, n = _spec_arrays(tuples)
    _weights_arg(weights, n, afterstate.device)
    delta_out = _out_arg(delta_out, (m,), torch.float32, afterstate.device, "delta_out")
    if m == 0:
        return delta_out
    lib = _lib.load()
    with torch.cuda.device(afterstate.device):
        rc = lib.ml2048_ntuple_td_update(afterstate.data_ptr(), target.data_ptr(), mask.data_ptr() if mask is not None else None,
                                         float(alpha), weights.data_ptr(), n, cells.ctypes.data, lens.ctypes.data, k,
                                         delta_out.data_ptr(), m, _stream(afterstate))
    _lib.check(rc, "ml2048_ntuple_td_update")
    return delta_out
