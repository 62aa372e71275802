"""Stand-alone device ops of the rollout path (thin wrappers over the C ABI, torch CUDA tensors in and out).

    sample_masked_categorical   _sample_action, policy/actor_critic.py:56-76
    gae_advantages              the recurrence of compute_gae, gae.py:50, :65-68
    encode_onehot               CNNEncoder.forward's input encoding, policy/_network.py:86-95
    valid_actions               _compute_valid_actions, game_numba.py:259-289
    afterstates                 all four moves of every board up to the spawn: _step_kernel + reward_fn, game_numba.py:93-134,
                                :408-504 at :728 (moved board, reward, "the move changes the board", optionally `merged`)
"""

from __future__ import annotations

from typing import Optional

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
