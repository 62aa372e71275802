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
    ntuple_expectimax           the expectimax move over such a network, one or two chance layers deep
    ntuple_tc_update            a temporal coherence batch update of such a network: per-weight step sizes
    ntuple_td_lambda_update,    delayed TD(lambda) / TC(lambda): the afterstate of h steps ago toward a lambda-return over
    ntuple_tc_lambda_update     the caller's ring of each game's last h + 1 afterstates, valued in one kernel
    ntuple_stages               every ntuple_* op takes ``stages=``: a multi-stage network, one weight set per stage of the
                                game, chosen by the board's largest tile
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


def _out_arg(t, shape: tuple, dtype, device, name: str) -> torch.Tensor:
    if t is None:
        return torch.empty(shape, dtype=dtype, device=device)
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous() and t.dtype == dtype and tuple(t.shape) == shape
            and t.device == device):
        raise ValueError(f"{name} must be a contiguous {dtype} tensor {shape} on {device}")
    return t


def _out_dict(out, keys, op: str) -> dict:
    """the ``out`` argument of an op that returns a dict of tensors: None or a dict holding any subset of ``keys``"""
    out = {} if out is None else out
    if not isinstance(out, dict):
        raise ValueError("out must be a dict of tensors")
    unknown = set(out) - set(keys)
    if unknown:
        raise ValueError(f"out has entries {op} does not write: {sorted(unknown)}")
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
    out = _out_dict(out, keys, "afterstates")
    _cuda(board, "board")
    m = board.shape[0]
    res = {k: _out_arg(out.get(k), (m,) + _AFTERSTATES[k][0], _AFTERSTATES[k][1], board.device, f"out[{k!r}]") for k in keys}
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


NTUPLE_MAX_STAGES = 8


def ntuple_stages(stages) -> tuple:
    """Check a multi-stage network's stage thresholds on the host and return them as a tuple of ints.

    S - 1 = 0..7 strictly ascending tile exponents in 1..15 (ints, not bools) give S = 1..8 stages; () is the single-stage
    network.  Raises ValueError otherwise.  With thresholds tau_1 < ... < tau_{S-1}, m(b) = max over the 16 cells of
    min(b[c], 15) (the index's own clamp) and stage(b) = #{k : tau_k <= m(b)}: an empty board is in stage 0, a byte >= 16
    counts as 15.  The weights are S * N float32 entries (N = sum 16^len), stage s's tables at s * N in the single-stage
    layout.  V(b) uses the tables of b's own stage (greedy: each afterstate's; expectimax: each leaf's; TD(lambda): each
    window board's), and every update writes the entries of x_0's stage.  Everything else is the single-stage op's, and
    S = 1 is that op bit for bit."""
    try:
        got = tuple(stages)
    except TypeError:
        raise ValueError(f"stages must be a sequence of tile exponents, got {stages!r}") from None
    if any(isinstance(t, bool) or not isinstance(t, (int, np.integer)) for t in got):
        raise ValueError(f"stages must be ints, got {stages!r}")
    got = tuple(int(t) for t in got)
    if len(got) > NTUPLE_MAX_STAGES - 1:
        raise ValueError(f"a network has at most {NTUPLE_MAX_STAGES} stages ({NTUPLE_MAX_STAGES - 1} thresholds), "
                         f"got {len(got)} thresholds")
    if any(t < 1 or t > 15 for t in got) or any(a >= b for a, b in zip(got, got[1:])):
        raise ValueError(f"stage thresholds are strictly ascending tile exponents in 1..15, got {got}")
    return got


def ntuple_num_weights(tuples, stages=()) -> int:
    """S * sum over the tuples of 16^len: the length of the network's one float32 weight tensor (S = len(stages) + 1)"""
    return (len(ntuple_stages(stages)) + 1) * sum(16 ** len(t) for t in ntuple_spec(tuples))


_SPEC_ARRAYS: dict = {}
_STAGE_ARRAYS: dict = {}


def _stage_array(stages):
    """(host threshold array u8 [S-1] or None, S) of the checked stages.  Every call checks ``stages``; the array is cached
    per checked tuple so that repeated calls do not build it again (the library reads it on the host, during the call)."""
    st = ntuple_stages(stages)
    got = _STAGE_ARRAYS.get(st)
    if got is None:
        got = (np.array(st, np.uint8) if st else None, len(st) + 1)
        if len(_STAGE_ARRAYS) < 64:
            _STAGE_ARRAYS[st] = got
    return got


def _network_args(tuples, stages):
    """(cells, len, K, stage thresholds or None, S, number of weights S * N) of a checked network"""
    cells, lens, k, n = _spec_arrays(tuples)
    tau, s = _stage_array(stages)
    return cells, lens, k, tau, s, s * n


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


def _weights_arg(weights: torch.Tensor, n: int, device, stages: int = 1) -> None:
    if not (isinstance(weights, torch.Tensor) and weights.is_cuda and weights.is_contiguous() and weights.dtype == torch.float32
            and weights.ndim == 1):
        raise ValueError("weights must be a contiguous 1-D float32 CUDA tensor")
    if weights.numel() != n:
        if stages > 1:
            raise ValueError(f"weights has {weights.numel()} entries, the tuples and {stages} stages need S * sum 16^len = {n}")
        raise ValueError(f"weights has {weights.numel()} entries, the tuples need sum 16^len = {n}")
    if weights.device != device:
        raise ValueError(f"weights is on {weights.device}, the boards on {device}")


def _promoted_arg(promoted, n: int, device) -> tuple:
    """() without marks, else (pointer,) of checked marks: a contiguous (N,) uint8 CUDA tensor on ``device``, 4-byte aligned"""
    if promoted is None:
        return ()
    if not (isinstance(promoted, torch.Tensor) and promoted.is_cuda and promoted.is_contiguous() and promoted.dtype == torch.uint8
            and tuple(promoted.shape) == (n,) and promoted.device == device):
        raise ValueError(f"promoted must be a contiguous uint8 ({n},) tensor on {device}")
    if promoted.data_ptr() % 4:
        raise ValueError("promoted must be 4-byte aligned (the marks are set with 32-bit atomics)")
    return (promoted.data_ptr(),)


def _entry(name: str, promoted: tuple) -> str:
    """the library entry of op ``name``: ml2048_staged_* without marks, ml2048_promoted_* with them"""
    return f"ml2048_{'promoted' if promoted else 'staged'}_{name}"


def ntuple_promoted_weights(weights: torch.Tensor, promoted: torch.Tensor, tuples, stages) -> torch.Tensor:
    """The S * N effective weights of a promoting network, a new tensor in the layout of ``weights``: W(0, e) = weights[e]
    and, for s >= 1, W(s, e) = weights[s * N + e] where bit s - 1 of ``promoted[e]`` is set, else W(s - 1, e).  A staged op
    on these weights gives what the op with ``promoted=promoted`` gives on ``weights``."""
    cells, lens, k, tau, s, n = _network_args(tuples, stages)
    _weights_arg(weights, n, getattr(weights, "device", None), s)
    _promoted_arg(promoted, n // s, weights.device)
    eff = weights.view(s, n // s).clone()
    for st in range(1, s):
        eff[st] = torch.where((promoted & (1 << (st - 1))) != 0, eff[st], eff[st - 1])
    return eff.view(-1)


def _ptr(a) -> Optional[int]:
    return None if a is None else a.ctypes.data


def _board_arg(board, name: str = "board") -> None:
    if not isinstance(board, torch.Tensor) or board.dtype not in (torch.uint8, torch.int8) or board.ndim != 2 or board.shape[1] != 16:
        raise ValueError(f"{name} must be uint8/int8 (M,16)")
    _cuda(board, name)


def ntuple_value(board: torch.Tensor, weights: torch.Tensor, tuples, *, out: Optional[torch.Tensor] = None,
                 stages=(), promoted: Optional[torch.Tensor] = None) -> torch.Tensor:
    """V(board) of an n-tuple network: (M,16) uint8/int8 boards -> (M,) float32.

    ``tuples``: the network's cells (see ``ntuple_spec``); ``weights``: its one float32 tensor of sum 16^len entries, tuple t's
    table after those of tuples 0..t-1.  V sums, for t = 0..K-1 and then each of the board's 8 symmetric images g = 0..7,
    ``weights[offset_t + sum_j min(image_g[cell_tj], 15) << 4j]`` as float32 adds from 0 in that order: bit-reproducible.
    Every byte gives an in-bounds index; tiles 2^16 and above share the entries of 2^15.  ``out``: a preallocated (M,)
    float32 tensor (CUDA-graph capture).  ``stages``: the thresholds of a multi-stage network (``ntuple_stages``); its
    ``weights`` hold S * sum 16^len entries and each board is valued with the tables of its own stage.

    ``promoted``: the marks of a multi-stage network with weight promotion (Jaskowski 2018), a contiguous (N,) uint8 CUDA
    tensor, N = sum 16^len for any S, or None (no promotion).  Bit s - 1 of ``promoted[e]`` is set once stage s's entry e has
    been written; every op then reads the effective weight W(s, e) = weights[s * N + e] if that bit is set, else W(s - 1, e)
    (W(0, e) = weights[e]), in the same float32 order as without marks (``ntuple_promoted_weights``).  The storage of an
    unmarked entry is never read.  With one stage the marks are neither read nor written."""
    _board_arg(board)
    cells, lens, k, tau, s, n = _network_args(tuples, stages)
    _weights_arg(weights, n, board.device, s)
    pm = _promoted_arg(promoted, n // s, board.device)
    m = board.shape[0]
    out = _out_arg(out, (m,), torch.float32, board.device, "out")
    if m == 0:
        return out
    lib = _lib.load()
    fn = _entry("value", pm)
    with torch.cuda.device(board.device):
        rc = getattr(lib, fn)(board.data_ptr(), weights.data_ptr(), n, cells.ctypes.data, lens.ctypes.data, k, _ptr(tau), s, *pm,
                              out.data_ptr(), m, _stream(board))
    _lib.check(rc, fn)
    return out


_NTUPLE_GREEDY = {"state": ((16,), torch.uint8), "reward": ((), torch.float32), "value": ((), torch.float32)}


def _move_outputs(out, specs: dict, action_dtype, board, op: str) -> dict:
    """the outputs of a move choice: "action" and ``specs`` (key -> (shape after M, dtype)), each ``out``'s tensor or a new one"""
    specs = {"action": ((), action_dtype), **specs}
    out = _out_dict(out, specs, op)
    m = board.shape[0]
    return {k: _out_arg(out.get(k), (m,) + shape, dtype, board.device, f"out[{k!r}]") for k, (shape, dtype) in specs.items()}


def ntuple_greedy(board: torch.Tensor, weights: torch.Tensor, tuples, *, reward_fn=None, action_dtype: torch.dtype = torch.int64,
                  out: Optional[dict] = None, stages=(), promoted: Optional[torch.Tensor] = None) -> dict:
    """The greedy afterstate move of every board under an n-tuple network, in one kernel.

    For every direction a that changes the board, q_a = reward_a + V(afterstate_a) in float32, with reward_a and afterstate_a
    exactly ``afterstates(board, reward_fn=reward_fn)``'s.  The largest q wins; NaN ranks as -inf; ties go to the smallest a.
    Returns a dict of CUDA tensors:

        "action"  (M,)    action_dtype (int64 or uint8)
        "state"   (M,16)  uint8    the chosen afterstate (no tile spawned)
        "reward"  (M,)    float32  its reward
        "value"   (M,)    float32  V(afterstate)

    A board without a valid move gets action 0, its own board, reward 0 and value 0 (so a TD target reward + value is 0).
    ``out``: preallocated tensors under the same keys (any subset), so that the call can be captured in a CUDA graph.
    ``stages``: a multi-stage network (``ntuple_stages``); each afterstate is valued with the tables of its own stage.
    ``promoted``: the network's promotion marks (``ntuple_value``), or None."""
    _board_arg(board)
    if action_dtype not in (torch.int64, torch.uint8):
        raise ValueError("action_dtype must be torch.int64 or torch.uint8")
    kind = reward_kind(reward_fn)
    cells, lens, k, tau, s, n = _network_args(tuples, stages)
    _weights_arg(weights, n, board.device, s)
    pm = _promoted_arg(promoted, n // s, board.device)
    m = board.shape[0]
    res = _move_outputs(out, _NTUPLE_GREEDY, action_dtype, board, "ntuple_greedy")
    if m == 0:
        return res
    act = res["action"].data_ptr()
    lib = _lib.load()
    fn = _entry("greedy", pm)
    with torch.cuda.device(board.device):
        rc = getattr(lib, fn)(board.data_ptr(), weights.data_ptr(), n, cells.ctypes.data, lens.ctypes.data, k, _ptr(tau), s, *pm, kind,
                              act if action_dtype == torch.uint8 else None, act if action_dtype == torch.int64 else None,
                              res["state"].data_ptr(), res["reward"].data_ptr(), res["value"].data_ptr(), m, _stream(board))
    _lib.check(rc, fn)
    return res


_NTUPLE_EXPECTIMAX = dict(_NTUPLE_GREEDY, q=((4,), torch.float32))


def ntuple_expectimax(board: torch.Tensor, weights: torch.Tensor, tuples, *, depth: int = 1, two_prob: float = 0.8, reward_fn=None,
                      action_dtype: torch.dtype = torch.int64, out: Optional[dict] = None, stages=(),
                      promoted: Optional[torch.Tensor] = None) -> dict:
    """The expectimax move of every board under an n-tuple network, ``depth`` (1 or 2) chance layers deep, in one kernel.

    Definition (every operation one float32 operation; after, r, valid as ``afterstates(board, reward_fn=reward_fn)`` gives
    them, V = ``ntuple_value``, p2 = float32(two_prob), p4 = 1 - p2 in float32):

        E(s, d)  chance node of afterstate s: for each empty cell c of s in ascending order
                 t_c = p2 * M(s + tile 2 at c, d) + p4 * M(s + tile 4 at c, d)  (an outcome of probability 0 is left out);
                 E = (t_c1 + t_c2 + ...) / n, added in that order starting from the first term
        M(b, d)  max over valid a of key(r(b,a) + (V(after(b,a)) if d == 1 else E(after(b,a), d - 1))), key(NaN) = -inf,
                 the smallest direction's key among equal keys; 0 for a board without a valid move
        q_a      r(b,a) + E(after(b,a), depth) for a valid a, -inf otherwise

    The action is the argmax of q with ``ntuple_greedy``'s rule (NaN ranks as -inf, ties go to the smallest direction).
    Depth 1 is "2-ply" expectimax in the literature.  The spawn model is VecGame's marginal law: a uniform empty cell, a 2
    with probability ``two_prob``.  VecGame ties 2-vs-4 to the cell within a table epoch; the search deliberately does not
    model that tie.  Returns a dict of CUDA tensors:

        "action"  (M,)    action_dtype (int64 or uint8)
        "state"   (M,16)  uint8    the chosen afterstate (no tile spawned)
        "reward"  (M,)    float32  its reward
        "value"   (M,)    float32  E(afterstate, depth)
        "q"       (M,4)   float32  q of every direction

    A board without a valid move gets action 0, its own board, reward 0, value 0 and q all -inf.  ``out``: preallocated
    tensors under the same keys (any subset), so that the call can be captured in a CUDA graph.  Cells must be 0..17.
    ``stages``: a multi-stage network (``ntuple_stages``); each leaf is valued with the tables of its own stage.
    ``promoted``: the network's promotion marks (``ntuple_value``), or None."""
    _board_arg(board)
    if action_dtype not in (torch.int64, torch.uint8):
        raise ValueError("action_dtype must be torch.int64 or torch.uint8")
    if isinstance(depth, bool) or depth not in (1, 2):
        raise ValueError(f"depth must be 1 or 2, got {depth!r}")
    try:
        p = float(two_prob)
    except (TypeError, ValueError):
        raise ValueError(f"two_prob must be a number in [0, 1], got {two_prob!r}") from None
    if not 0.0 <= p <= 1.0:
        raise ValueError(f"two_prob must be in [0, 1], got {two_prob!r}")
    kind = reward_kind(reward_fn)
    cells, lens, k, tau, s, n = _network_args(tuples, stages)
    _weights_arg(weights, n, board.device, s)
    pm = _promoted_arg(promoted, n // s, board.device)
    m = board.shape[0]
    res = _move_outputs(out, _NTUPLE_EXPECTIMAX, action_dtype, board, "ntuple_expectimax")
    if m == 0:
        return res
    act = res["action"].data_ptr()
    lib = _lib.load()
    fn = _entry("expectimax", pm)
    with torch.cuda.device(board.device):
        rc = getattr(lib, fn)(board.data_ptr(), weights.data_ptr(), n, cells.ctypes.data, lens.ctypes.data, k, _ptr(tau), s, *pm, kind,
                              int(depth), p, act if action_dtype == torch.uint8 else None,
                              act if action_dtype == torch.int64 else None, res["state"].data_ptr(), res["reward"].data_ptr(),
                              res["value"].data_ptr(), res["q"].data_ptr(), m, _stream(board))
    _lib.check(rc, fn)
    return res


def _coherence_args(coherence, accum, n: int, device) -> tuple[int, int]:
    """checks of TC's ``coherence`` and ``accum``; returns their pointers"""
    for name, t in (("coherence", coherence), ("accum", accum)):
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous() and t.dtype == torch.float32
                and tuple(t.shape) == (n, 2) and t.device == device):
            raise ValueError(f"{name} must be a contiguous float32 ({n}, 2) tensor on {device}")
    return coherence.data_ptr(), accum.data_ptr()


def _target_update(op: str, afterstate, target, weights, tuples, stages, promoted, alpha, mask, delta_out, tc=None) -> torch.Tensor:
    """ntuple_td_update (tc None) and ntuple_tc_update (tc = (coherence, accum)) through the library entry of ``op``
    (``_entry``)"""
    _board_arg(afterstate, "afterstate")
    m = afterstate.shape[0]
    _cuda(target, "target")
    if target.dtype != torch.float32 or tuple(target.shape) != (m,):
        raise ValueError(f"target must be float32 ({m},)")
    if mask is not None:
        _cuda(mask, "mask")
        if mask.dtype not in (torch.bool, torch.uint8) or tuple(mask.shape) != (m,):
            raise ValueError(f"mask must be bool/uint8 ({m},)")
    cells, lens, k, tau, s, n = _network_args(tuples, stages)
    _weights_arg(weights, n, afterstate.device, s)
    tc_ptrs = () if tc is None else _coherence_args(*tc, n, afterstate.device)
    pm = _promoted_arg(promoted, n // s, afterstate.device)
    delta_out = _out_arg(delta_out, (m,), torch.float32, afterstate.device, "delta_out")
    if m == 0:
        return delta_out
    lib = _lib.load()
    fn = _entry(op, pm)
    with torch.cuda.device(afterstate.device):
        rc = getattr(lib, fn)(afterstate.data_ptr(), target.data_ptr(), mask.data_ptr() if mask is not None else None, float(alpha),
                              weights.data_ptr(), *tc_ptrs, n, cells.ctypes.data, lens.ctypes.data, k, _ptr(tau), s, *pm,
                              delta_out.data_ptr(), m, _stream(afterstate))
    _lib.check(rc, fn)
    return delta_out


def ntuple_td_update(afterstate: torch.Tensor, target: torch.Tensor, weights: torch.Tensor, tuples, *, alpha: float,
                     mask: Optional[torch.Tensor] = None, delta_out: Optional[torch.Tensor] = None, stages=(),
                     promoted: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One synchronous batch of TD(0) updates of an n-tuple network, in place on ``weights``; returns delta (M,) float32.

    Phase 1: delta_i = alpha * (target_i - V(afterstate_i)) with the weights as they were before the call, 0 for a game
    whose ``mask`` byte is 0 (``mask``: (M,) bool/uint8, None = every game).  Phase 2: every entry of every masked-in game,
    8 per tuple, gets += delta_i.  Phase 2 adds with float atomics, so the order of the adds that several games make to one
    entry is unspecified: the weights are reproducible only up to the fp32 rounding of that order.  delta is deterministic.
    ``delta_out``: a preallocated (M,) float32 tensor (CUDA-graph capture).  ``stages``: a multi-stage network
    (``ntuple_stages``); V(afterstate_i) and the update use the tables of afterstate_i's stage.

    ``promoted``: the marks of a network with weight promotion (``ntuple_value``), updated in place.  delta is computed with
    the effective weights before the call; then every masked-in game whose afterstate is in a stage s >= 1 (whatever its
    delta, 0 included) promotes each of its entries e whose mark of (s, e) is clear: weights[s * N + e] = W(s - 1, e), and
    the mark is set.  Promotion changes no effective weight.  Phase 2 then adds to the entries of the afterstate's stage."""
    return _target_update("td_update", afterstate, target, weights, tuples, stages, promoted, alpha, mask, delta_out)


def ntuple_tc_update(afterstate: torch.Tensor, target: torch.Tensor, weights: torch.Tensor, coherence: torch.Tensor,
                     accum: torch.Tensor, tuples, *, alpha: float, mask: Optional[torch.Tensor] = None,
                     delta_out: Optional[torch.Tensor] = None, stages=(), promoted: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One synchronous batch of temporal coherence (TC) updates of an n-tuple network, in place on ``weights`` and
    ``coherence``; returns delta (M,) float32.

    Every weight has its own step size beta_j = |E_j| / A_j, with ``coherence[j] = (E_j, A_j)`` the running sum of the errors
    applied to entry j and of their absolute values (Jaskowski 2018).  Every operation is one float32 operation:

    1. delta_i = alpha * (target_i - V(afterstate_i)) with the weights as they were before the call, 0 for a game whose
       ``mask`` byte is 0 (``mask``: (M,) bool/uint8, None = every game) -- ``ntuple_td_update``'s delta bit for bit;
    2. for every masked-in game and each of its 8K entries j (twice if the game hits j twice): dE_j += delta_i,
       dA_j += |delta_i|, float atomics into ``accum`` (order within one entry unspecified, subnormals flushed);
    3. for every entry with dA_j != 0 (NaN counts as non-zero), with E_j and A_j as they were before the call:
       beta_j = 1 if A_j == 0 else |E_j| / A_j;  w_j += beta_j * dE_j;  E_j += dE_j;  A_j += dA_j.
       Entries with dA_j == 0 stay as they are, bit for bit.

    E and A sum alpha-scaled errors: with a constant alpha, beta is the same as for unscaled errors; a changing alpha weights
    older errors by the alpha they had.  ``coherence`` and ``accum``: contiguous float32 (N, 2) tensors on the weights'
    device; ``accum`` is scratch that must be all zero and is left all zero.  ``delta_out``: a preallocated (M,) float32
    tensor (CUDA-graph capture).  ``stages``: a multi-stage network (``ntuple_stages``); ``weights`` has S * N entries,
    ``coherence`` and ``accum`` are (S * N, 2), and afterstate_i's value and update use the entries of its stage.
    ``promoted``: as for ``ntuple_td_update``; a promoted entry's coherence is set to (0, 0), so its first TC step has
    beta = 1."""
    return _target_update("tc_update", afterstate, target, weights, tuples, stages, promoted, alpha, mask, delta_out,
                          (coherence, accum))


NTUPLE_LAMBDA_MAX_HORIZON = 16


def _lambda_update(op: str, after_ring, reward_ring, ended_ring, newest, weights, tuples, stages, promoted, alpha, lam, mask,
                   delta_out, tc=None) -> torch.Tensor:
    """ntuple_td_lambda_update (tc None) and ntuple_tc_lambda_update (tc = (coherence, accum)) through the library entry of
    ``op`` (``_entry``)"""
    if not (isinstance(after_ring, torch.Tensor) and after_ring.dtype in (torch.uint8, torch.int8) and after_ring.ndim == 3
            and after_ring.shape[2] == 16):
        raise ValueError("after_ring must be uint8/int8 (h+1, M, 16)")
    slots, m = after_ring.shape[0], after_ring.shape[1]
    h = slots - 1
    if not 1 <= h <= NTUPLE_LAMBDA_MAX_HORIZON:
        raise ValueError(f"after_ring holds h + 1 = {slots} slots: the horizon h must be 1..{NTUPLE_LAMBDA_MAX_HORIZON}")
    if isinstance(newest, bool) or not isinstance(newest, int) or not 0 <= newest <= h:
        raise ValueError(f"newest must be an int slot 0..{h}, got {newest!r}")
    try:
        lam = float(lam)
    except (TypeError, ValueError):
        raise ValueError(f"lam must be a number in [0, 1], got {lam!r}") from None
    if not 0.0 <= lam <= 1.0:
        raise ValueError(f"lam must be in [0, 1], got {lam!r}")
    _cuda(after_ring, "after_ring")
    dev = after_ring.device
    for name, t, dtypes in (("reward_ring", reward_ring, (torch.float32,)), ("ended_ring", ended_ring, (torch.bool, torch.uint8))):
        _cuda(t, name)
        if t.dtype not in dtypes or tuple(t.shape) != (slots, m) or t.device != dev:
            raise ValueError(f"{name} must be {'/'.join(str(d) for d in dtypes)} ({slots}, {m}) on {dev}")
    if mask is not None:
        _cuda(mask, "mask")
        if mask.dtype not in (torch.bool, torch.uint8) or tuple(mask.shape) != (m,) or mask.device != dev:
            raise ValueError(f"mask must be bool/uint8 ({m},) on {dev}")
    cells, lens, k, tau, s, n = _network_args(tuples, stages)
    _weights_arg(weights, n, dev, s)
    tc_ptrs = () if tc is None else _coherence_args(*tc, n, dev)
    pm = _promoted_arg(promoted, n // s, dev)
    delta_out = _out_arg(delta_out, (m,), torch.float32, dev, "delta_out")
    if m == 0:
        return delta_out
    lib = _lib.load()
    fn = _entry(op, pm)
    with torch.cuda.device(dev):
        rc = getattr(lib, fn)(after_ring.data_ptr(), reward_ring.data_ptr(), ended_ring.data_ptr(), h, newest, lam,
                              mask.data_ptr() if mask is not None else None, float(alpha), weights.data_ptr(), *tc_ptrs, n,
                              cells.ctypes.data, lens.ctypes.data, k, _ptr(tau), s, *pm, delta_out.data_ptr(), m, _stream(after_ring))
    _lib.check(rc, fn)
    return delta_out


def ntuple_td_lambda_update(after_ring: torch.Tensor, reward_ring: torch.Tensor, ended_ring: torch.Tensor, newest: int,
                            weights: torch.Tensor, tuples, *, alpha: float, lam: float, mask: Optional[torch.Tensor] = None,
                            delta_out: Optional[torch.Tensor] = None, stages=(),
                            promoted: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One synchronous batch of delayed TD(lambda) updates of an n-tuple network (Jaskowski 2018), in place on ``weights``:
    each game's afterstate of h learner steps ago moves toward a lambda-return truncated at h.  Returns delta (M,) float32.

    Game i's window is x_0 ... x_h: x_0 the afterstate being updated, chosen h learner steps ago; x_h the one chosen this
    step; rho_k (k = 1..h) the reward of the move that produced x_k; e_k (k = 0..h-1) = 1 when the environment step after
    x_k was chosen ended the game; V_k = V(x_k) (``ntuple_value``) with the weights as they are before the call.  With
    lf = float32(lam) and c = 1 - lf in float32, every operation one float32 operation:

        R_{h-1} = e_{h-1} ? 0 : rho_h + V_h
        R_k     = e_k     ? 0 : (rho_{k+1} + c * V_{k+1}) + lf * R_{k+1}      for k = h-2 ... 0
        delta   = alpha * (R_0 - V_0)                                         (0 for a game whose ``mask`` byte is 0)

    then ``ntuple_td_update``'s phase 2 on x_0's entries (float atomics).  h = 1 is ``ntuple_td_update``'s delta with
    target = (0 if e_0 else rho_1 + V_1), bit for bit.  Values after the first end in a window are not looked up.

    The ring is the caller's: ``after_ring`` (h+1, M, 16) uint8/int8, ``reward_ring`` (h+1, M) float32, ``ended_ring``
    (h+1, M) bool/uint8, all contiguous on one device, h = ``after_ring.shape[0] - 1`` in 1..16.  ``newest`` is the slot of
    x_h; x_k is in slot (newest - (h - k)) mod (h + 1), and ``ended_ring[newest]`` is not read.  ``mask``: (M,) bool/uint8,
    None = every game.  ``delta_out``: a preallocated (M,) float32 tensor (CUDA-graph capture).  ``stages``: a multi-stage
    network (``ntuple_stages``); each V_k uses the tables of x_k's stage, and the update writes the entries of x_0's stage.
    ``promoted``: as for ``ntuple_td_update``: every V_k reads the effective weights, and x_0's entries are promoted before
    the adds."""
    return _lambda_update("lambda_td_update", after_ring, reward_ring, ended_ring, newest, weights, tuples, stages, promoted, alpha,
                          lam, mask, delta_out)


def ntuple_tc_lambda_update(after_ring: torch.Tensor, reward_ring: torch.Tensor, ended_ring: torch.Tensor, newest: int,
                            weights: torch.Tensor, coherence: torch.Tensor, accum: torch.Tensor, tuples, *, alpha: float,
                            lam: float, mask: Optional[torch.Tensor] = None,
                            delta_out: Optional[torch.Tensor] = None, stages=(),
                            promoted: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One synchronous batch of delayed TC(lambda) updates, in place on ``weights`` and ``coherence``; returns delta (M,)
    float32.  delta is ``ntuple_td_lambda_update``'s (the same window, ring, definition and arguments); the update of x_0's
    entries is then ``ntuple_tc_update``'s phases 2 and 3: {dE, dA} += {delta, |delta|} into ``accum``, and w += beta * dE,
    beta = |E| / A (1 where A = 0), {E, A} += {dE, dA} for every entry with dA != 0.  ``coherence`` and ``accum``: contiguous
    float32 (N, 2) tensors on the ring's device; ``accum`` must be all zero and is left all zero.  ``stages``: as for
    ``ntuple_td_lambda_update``, with ``coherence`` and ``accum`` (S * N, 2).  ``promoted``: as for ``ntuple_tc_update``."""
    return _lambda_update("lambda_tc_update", after_ring, reward_ring, ended_ring, newest, weights, tuples, stages, promoted, alpha,
                          lam, mask, delta_out, (coherence, accum))
