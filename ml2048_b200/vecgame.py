"""
``VecGame`` -- the B200-native drop-in for the reference's vectorised 2048 environment.

Same class surface as the reference (reference: src/ml2048/game_numba.py:522-698):

    VecGame(size, reward_fn=None, *, two_prob=0.8, reuse_state=False)
    .reset(seed)  .prepare() -> (indices,)  .observations() -> (board, valid)
    .step(actions) -> VecStepResult  .summary()   attributes: ._size ._data ._game_count

but all per-game state lives in HBM as struct-of-arrays torch CUDA tensors and every per-step
computation is a hand-written sm_100a kernel behind the C ABI of ``include/ml2048_b200.h``.
Host code here only (a) draws the reference's state-independent host random numbers
(``host_rng.py``), (b) passes pointers, (c) copies results to the host when the caller asked for
NumPy.  There is no CPU implementation of the game in this package.

Keyword-only extras (not in the reference):
    device        CUDA device (default: current)
    output        "numpy" (default, drop-in for the unmodified VecRunner: results are host arrays)
                  or "torch" (results are views of the live CUDA tensors; no host copies)
    rng_mode      "replay" (default; bit-exact with the reference) or "philox" (counter-based, no tables)
    onehot        None | "f32" | "bf16" | "u8": fuse the CNN's one-hot board encoding
                  (policy/_network.py:86-95) into step()/prepare(); read it with observations_onehot()
    track_merged  keep the per-game ``merged`` array (default True, as the reference)
    slot_base     global slot of game 0 (multi-GPU sharding: results do not depend on the shard count)
    sync_free     prepare() returns (None,) and never synchronises (CUDA-graph / benchmark loops)
"""

from __future__ import annotations

import ctypes as C
import os
from typing import Any, Optional

import numpy as np
import torch

from . import _lib
from .host_rng import RAND_ROWS, make_schedule
from .rewards import reward_kind

try:  # the raw-handle accessor is private but ~10x cheaper than building a Stream object per call
    _raw_stream = torch._C._cuda_getCurrentRawStream
except AttributeError:  # pragma: no cover - older/newer torch without it

    def _raw_stream(index: int) -> int:
        return torch.cuda.current_stream(index).cuda_stream


try:  # torch.cuda.current_device() minus its lazy-init bookkeeping (this runs five times per runner step)
    _current_device = torch._C._cuda_getDevice
except AttributeError:  # pragma: no cover
    _current_device = torch.cuda.current_device

_ONEHOT = {
    None: (_lib.ONEHOT_NONE, None),
    "f32": (_lib.ONEHOT_F32, torch.float32),
    "bf16": (_lib.ONEHOT_BF16, torch.bfloat16),
    "u8": (_lib.ONEHOT_U8, torch.uint8),
}

# the reference's record layout (game_numba.py:537-551), used by the `_data` compatibility view
DATA_DTYPE = np.dtype(
    [
        ("id", np.int32, ()),
        ("step", np.int32, ()),
        ("score", np.float32, ()),
        ("reward", np.float32, ()),
        ("board", np.uint8, (16,)),
        ("merged", np.uint8, (16,)),
        ("valid_actions", np.uint8, (4,)),
        ("terminated", np.uint8, ()),
        ("invalid", np.uint8, ()),
        ("_padding", np.uint8, 10),
    ],
    align=True,
)


class VecStepResult(dict):
    """The 10-key result of ``step()`` (game_numba.py:507-519, 687-698).

    In the reference the values are views of live arrays.  Here they are fetched from the live device
    tensors when a key is first read (NumPy mode: one D2H copy of exactly that field; torch mode: a
    view of the CUDA tensor), which gives the same "current contents" semantics without copying
    fields nobody reads."""

    KEYS = ("state", "valid_actions", "merged", "step", "reward", "score", "terminated", "invalid", "prev_state",
            "prev_valid_actions")

    def __init__(self, env: "VecGame"):
        super().__init__()
        self._env = env

    def __missing__(self, key: str):
        if key not in self.KEYS:
            raise KeyError(key)
        value = self._env._fetch(key)
        self[key] = value
        return value

    def __contains__(self, key: object) -> bool:
        return key in self.KEYS

    def keys(self):
        return list(self.KEYS)

    def items(self):
        return [(k, self[k]) for k in self.KEYS]

    def values(self):
        return [self[k] for k in self.KEYS]

    def __iter__(self):
        return iter(self.KEYS)

    def __len__(self) -> int:
        return len(self.KEYS)


class _DataView:
    """Stand-in for the reference's structured array ``VecGame._data`` (game_numba.py:571).

    ``view["id"]`` copies one field to the host; ``view[slot]`` / ``view[indices]`` gathers whole
    64-byte records (replay.py:147-151 reads ``game._data[slot]["id"].item()``)."""

    def __init__(self, env: "VecGame"):
        self._env = env

    def __len__(self) -> int:
        return self._env._size

    @property
    def dtype(self) -> np.dtype:
        return DATA_DTYPE

    # Whole-record lookups are served from a HOST copy of the state arena when that is cheap: the pinned mirror the
    # NumPy drop-in mode fills at every prepare()/step() of a small batch, or (up to _SNAPSHOT_MAX_GAMES) one copy +
    # one synchronisation made on the first lookup after the state last changed.  ReplayRecorder.on_prepared reads
    # ``data[slot]["id"].item()`` in a Python loop over the reset slots (replay.py:147-151): 65 536 lookups at
    # eval_perf.py's first prepare() cost one 3.5 MB copy instead of 65 536 x nine gathers.  Larger batches gather the
    # requested records on the device and bring them over with ONE copy.
    _SNAPSHOT_MAX_GAMES = 1 << 20

    def _host_views(self):
        env = self._env
        if env._mirror_epoch == env._state_epoch and env._arena_host is not None:
            return env._mirror
        if env._size <= self._SNAPSHOT_MAX_GAMES:
            return env._mirror_to_host()
        return None

    @staticmethod
    def _normalise_key(key: Any, size: int):
        """-> (index array or None for 'everything', scalar?) without materialising arange(size) for a single slot."""
        if isinstance(key, (int, np.integer)):
            k = int(key)
            if k < -size or k >= size:
                raise IndexError(f"index {k} is out of bounds for {size} games")
            return np.asarray([k % size], dtype=np.int64), True
        if isinstance(key, slice):
            if key == slice(None):
                return None, False
            return np.arange(*key.indices(size), dtype=np.int64), False
        if isinstance(key, torch.Tensor):
            key = key.cpu().numpy()
        key = np.asarray(key)
        if key.dtype == np.bool_:
            return np.flatnonzero(key).astype(np.int64), False
        idx = key.astype(np.int64).reshape(-1)
        if idx.size and (idx.min() < -size or idx.max() >= size):
            raise IndexError(f"index out of bounds for {size} games")
        return np.where(idx < 0, idx + size, idx), False

    def __getitem__(self, key: Any):
        env = self._env
        if isinstance(key, str):
            name = {"board": "state"}.get(key, key)
            if key == "id":
                return env._to_host(env._id)
            if key == "_padding":
                return np.zeros((env._size, 10), np.uint8)
            return env._fetch(name, force_host=True)
        idx, scalar = self._normalise_key(key, env._size)
        cur = env._cur
        views = self._host_views()
        if views is not None:
            take = (lambda a: a.copy()) if idx is None else (lambda a: a[idx])
            n = env._size if idx is None else idx.size
            rec = np.zeros((n,), dtype=DATA_DTYPE)
            rec["id"] = take(views["_id"])
            rec["step"] = take(views["_step"])
            rec["score"] = take(views["_score"])
            rec["reward"] = take(views["_reward"])
            rec["board"] = take(views["_board"][cur])
            if env._merged is not None:
                rec["merged"] = take(views["_merged"])
            rec["valid_actions"] = take(views["_valid"][cur])
            rec["terminated"] = take(views["_terminated_padded"][: env._size])
            rec["invalid"] = take(views["_invalid"])
            return rec[0] if scalar else rec
        # large batch: gather the records on the device into one packed buffer, ONE copy to the host
        if idx is None:
            idx = np.arange(env._size, dtype=np.int64)
        didx = torch.from_numpy(idx).to(env.device)
        n = idx.size
        packed = torch.zeros((n, DATA_DTYPE.itemsize), dtype=torch.uint8, device=env.device)

        def put(field: str, t: torch.Tensor) -> None:
            off = DATA_DTYPE.fields[field][1]
            raw = t.index_select(0, didx).contiguous().view(torch.uint8).reshape(n, -1)
            packed[:, off:off + raw.shape[1]] = raw

        put("id", env._id)
        put("step", env._step_score.view(torch.int32)[:, 0])
        put("score", env._step_score.view(torch.int32)[:, 1])
        put("reward", env._reward)
        put("board", env._board[cur])
        if env._merged is not None:
            put("merged", env._merged)
        put("valid_actions", env._valid[cur])
        put("terminated", env._terminated)
        put("invalid", env._invalid)
        rec = packed.cpu().numpy().view(DATA_DTYPE).reshape(n)
        return rec[0] if scalar else rec

    def copy(self) -> np.ndarray:
        return self[:]


class VecGame:
    """Vectorised 2048 on one B200.  See the module docstring."""

    _RAND_SIZE: int = RAND_ROWS
    _DATA_DTYPE = DATA_DTYPE

    def __init__(
        self,
        size: int,
        reward_fn: Any = None,
        *,
        two_prob: float = 0.8,
        reuse_state: bool = False,
        device: Any = None,
        output: str = "numpy",
        rng_mode: str = "replay",
        onehot: Optional[str] = None,
        track_merged: bool = True,
        slot_base: int = 0,
        sync_free: bool = False,
    ):
        if size <= 0:
            raise ValueError(f"size={size}")  # game_numba.py:561-562
        if output not in ("numpy", "torch"):
            raise ValueError(f"output={output!r}")
        if rng_mode not in ("replay", "philox"):
            raise ValueError(f"rng_mode={rng_mode!r}")
        if onehot not in _ONEHOT:
            raise ValueError(f"onehot={onehot!r}")
        self._lib = _lib.load()  # raises if the CUDA library is missing: no fallback
        if not torch.cuda.is_available():
            raise RuntimeError("ml2048_b200.VecGame needs a CUDA device (there is no CPU fallback)")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise ValueError(f"device={device!r}: ml2048_b200 runs on CUDA only")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())

        self._size = int(size)
        self._two_prob = float(two_prob)
        self._reuse_state = reuse_state  # stored and unused, like the reference (game_numba.py:569)
        self._reward_fn = reward_fn
        self._reward_kind = reward_kind(reward_fn)
        self._output = output
        self._rng_mode = _lib.RNG_REPLAY if rng_mode == "replay" else _lib.RNG_PHILOX
        self._onehot_kind, onehot_dtype = _ONEHOT[onehot]
        self._slot_base = int(slot_base)
        self._sync_free = bool(sync_free)

        m, dev = self._size, self.device
        pad = (m + 15) // 16 * 16
        with torch.cuda.device(dev):
            # All per-game state the reference's callers can read lives in ONE arena (sub-buffers 256-byte aligned), so
            # that the NumPy drop-in mode can mirror it to the host with a single copy (see _mirror_to_host).
            layout = [("_reset_count_dev", torch.int64, (1,)), ("_game_count_dev", torch.int64, (1,)),  # count survives reset(), :582
                      ("_reset_indices_dev", torch.int64, (m,)), ("_board", torch.uint8, (2, m, 16)),
                      ("_valid", torch.uint8, (2, m, 4)), ("_id", torch.int32, (m,)),
                      ("_step_score", torch.int32, (m, 2)),  # {step, score} records: one stream for the kernels (ml2048_b200.h)
                      ("_reward", torch.float32, (m,)),
                      ("_terminated_padded", torch.uint8, (pad,)), ("_invalid", torch.uint8, (m,))]
            if track_merged:
                layout.append(("_merged", torch.uint8, (m, 16)))
            offsets, total = {}, 0
            for name, dtype, shape in layout:
                nbytes = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
                offsets[name] = (total, nbytes, dtype, shape)
                total += (nbytes + 255) // 256 * 256
            self._arena = torch.zeros((total,), dtype=torch.uint8, device=dev)
            self._arena_layout = offsets
            self._arena_host = None  # pinned mirror, allocated on first use
            self._state_epoch = 0    # bumped by everything that changes device state; the host mirror remembers its own
            self._mirror_epoch = -1
            for name, (off, nbytes, dtype, shape) in offsets.items():
                setattr(self, name, self._arena[off:off + nbytes].view(dtype).view(shape))
            self._terminated = self._terminated_padded[:m]
            # strided views of the records, like the reference's own views into its record array (game_numba.py:687-698)
            self._step = self._step_score[:, 0]
            self._score = self._step_score[:, 1].view(torch.float32)
            if not track_merged:
                self._merged = None
            self._onehot = torch.zeros((m, 16, 16), dtype=onehot_dtype, device=dev) if onehot_dtype is not None else None
            self._actions_out = torch.zeros((m,), dtype=torch.uint8, device=dev)
            # table ring: slot s holds [0] the reference's randperm table and [1] the same table in inverse
            # ("rank key") form.  Eager calls use one slot; a pre-drawn device schedule uses one slot per refresh.
            self._table_slots = 1
            self._tables_dev = torch.zeros((self._table_slots, 2, RAND_ROWS, 16), dtype=torch.uint8, device=dev)
            self._table_slot = 0
            self._sched_dev = None                       # int64 (L, 4): ml2048_sched_entry[L]
            self._sched_cursor_dev = torch.zeros((2,), dtype=torch.int64, device=dev)  # ping-pong like the boards
            self._id_offset_dev = torch.zeros((1,), dtype=torch.int64, device=dev)
            n_scratch = int(self._lib.ml2048_prepare_scratch_ints(m))
            self._scratch = torch.zeros((n_scratch,), dtype=torch.int32, device=dev)
            self._stats_dev = torch.zeros((_lib.STATS_REPLICAS, _lib.STATS_WORDS), dtype=torch.int64, device=dev)
        self._cur = 0
        self._host: dict[str, torch.Tensor] = {}  # pinned staging buffers, one per fetched field
        self._dev_index = self.device.index
        self._guard = VecGame._DeviceGuard(self._dev_index)
        # raw pointers of the ping-pong buffers (creating tensor views per call costs microseconds)
        self._board_ptr = (self._board[0].data_ptr(), self._board[1].data_ptr())
        self._valid_ptr = (self._valid[0].data_ptr(), self._valid[1].data_ptr())
        self._cursor_ptr = (self._sched_cursor_dev.data_ptr(), self._sched_cursor_dev.data_ptr() + 8)

        # host copies of the random tables, as in the reference (game_numba.py:577-580)
        self._randperm = np.empty((RAND_ROWS, 16), dtype=np.uint8)
        self._randfloat = np.empty((RAND_ROWS,), dtype=np.float32)
        self._tables_pin = None  # pinned staging ring for table uploads, allocated on first use
        self._record_active = False
        self._keep_record = None
        self._obs_cache = None
        self._sched_len = 0   # entries of the device-resident schedule (0 = eager mode: host draws per call)
        self._sched_pos = 0   # entries consumed so far (host mirror of the device cursor)
        self._rand_step = 0
        self._two_mask = 0
        self._two_threshold = int(self._lib.ml2048_two_threshold(self._two_prob))
        self._philox_seed = 0
        self._philox_counter = 0
        self._schedule: Any = None
        self._dist_group = None
        self._dist_rank = 0
        self._dist_world = 1
        self._id_bound = None
        self._skip_id_check = False
        self._reset_rank = None

        self._step_args = _lib.StepArgs()
        self._prep_args = _lib.PrepareArgs()
        self._init_args()
        self.reset()

    # ------------------------------------------------------------------------------------------
    # plumbing
    # ------------------------------------------------------------------------------------------

    @staticmethod
    def _p(t: Optional[torch.Tensor]) -> Optional[int]:
        return None if t is None else t.data_ptr()

    def _stream(self) -> int:
        return _raw_stream(self._dev_index)

    class _DeviceGuard:
        """Cheap `with torch.cuda.device(...)`: does nothing when the environment's device is already current."""

        __slots__ = ("_want", "_prev")

        def __init__(self, index: int):
            self._want = index
            self._prev = -1

        def __enter__(self):
            cur = _current_device()
            if cur != self._want:
                self._prev = cur
                torch.cuda.set_device(self._want)

        def __exit__(self, *exc):
            if self._prev >= 0:
                torch.cuda.set_device(self._prev)
                self._prev = -1

    def _init_args(self) -> None:
        a = self._step_args
        a.struct_size = C.sizeof(_lib.StepArgs)
        a.reward_kind = self._reward_kind
        a.rng_mode = self._rng_mode
        a.onehot_dtype = self._onehot_kind
        a.num_games = self._size
        a.slot_base = self._slot_base
        a.step = self._p(self._step)
        a.score = self._p(self._score)
        a.reward = self._p(self._reward)
        a.terminated = self._p(self._terminated_padded)
        a.invalid = self._p(self._invalid)
        a.merged = self._p(self._merged)
        a.onehot_out = self._p(self._onehot)
        a.two_threshold = self._two_threshold
        a.stats = self._p(self._stats_dev)
        p = self._prep_args
        p.struct_size = C.sizeof(_lib.PrepareArgs)
        p.rng_mode = self._rng_mode
        p.onehot_dtype = self._onehot_kind
        p.num_games = self._size
        p.slot_base = self._slot_base
        p.id = self._p(self._id)
        p.step = self._p(self._step)
        p.score = self._p(self._score)
        p.reward = self._p(self._reward)
        p.terminated = self._p(self._terminated_padded)
        p.invalid = self._p(self._invalid)
        p.merged = self._p(self._merged)
        p.onehot = self._p(self._onehot)
        p.two_threshold = self._two_threshold
        p.game_count = self._p(self._game_count_dev)
        p.id_offset = None
        p.reset_count = self._p(self._reset_count_dev)
        p.reset_indices = self._p(self._reset_indices_dev)
        p.scratch = self._p(self._scratch)

    def _pinned(self, name: str, t: torch.Tensor) -> torch.Tensor:
        buf = self._host.get(name)
        if buf is None or buf.shape != t.shape or buf.dtype != t.dtype:
            buf = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            self._host[name] = buf
        return buf

    def _to_host(self, t: torch.Tensor, key: Optional[str] = None) -> np.ndarray:
        """D2H through a pinned staging buffer owned by this environment (reused per field)."""
        buf = self._pinned(key or f"_anon{t.data_ptr()}", t)
        buf.copy_(t, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return buf.numpy()

    # NumPy (drop-in) mode, small batches: a runner step is dominated by the ~12 us each host<->device round trip
    # costs, so prepare() and step() mirror the WHOLE state arena to the host with one copy and one sync instead
    # of one copy + sync per field.  Large batches stay lazy: there the copies are PCIe-bandwidth bound.
    _EAGER_HOST_MAX_GAMES = 1 << 15
    # Medium batches: still latency-sensitive, but mirroring everything would waste bandwidth: the fields the reference's
    # callers read (runner.py:165, replay.py:170-173, run_train3.py:138-149) are copied together behind one synchronisation.
    _BATCHED_HOST_MAX_GAMES = 1 << 20
    _COMMON_FIELDS = ("state", "valid_actions", "prev_state", "prev_valid_actions", "reward", "score", "step", "terminated")

    def _fetch_many(self, keys) -> dict[str, np.ndarray]:
        """Several per-field D2H copies behind ONE synchronisation."""
        stream = torch.cuda.current_stream(self.device)
        bufs = {}
        for k in keys:
            t = self._device_field(k)
            buf = self._pinned(k, t)
            buf.copy_(t, non_blocking=True)
            bufs[k] = buf
        stream.synchronize()
        return {k: b.numpy() for k, b in bufs.items()}

    def _mirror_to_host(self) -> dict[str, np.ndarray]:
        """One D2H copy of the state arena into its pinned host mirror; returns NumPy views of the mirror by name."""
        if self._arena_host is None:
            self._arena_host = torch.empty(self._arena.shape, dtype=torch.uint8, pin_memory=True)
            flat = self._arena_host.numpy()
            views = {}
            for name, (off, nbytes, dtype, shape) in self._arena_layout.items():
                npdt = {torch.int64: np.int64, torch.int32: np.int32, torch.float32: np.float32, torch.uint8: np.uint8}[dtype]
                views[name] = flat[off:off + nbytes].view(npdt).reshape(shape)
            views["_step"] = views["_step_score"][:, 0]
            views["_score"] = views["_step_score"][:, 1].view(np.float32)
            self._mirror = views
            self._arena_copy = (self._arena_host.data_ptr(), self._arena.data_ptr(), self._arena.numel())
        # (the library's own copy + wait: a torch copy_ + current_stream().synchronize() costs ~15 us of host time per call,
        # more than the kernels of a 2048-game step take)
        stream = self._stream()
        with self._guard:
            dst, src, nbytes = self._arena_copy
            _lib.check(self._lib.ml2048_copy_async(dst, src, nbytes, stream), "ml2048_copy_async")
            _lib.check(self._lib.ml2048_stream_wait(stream), "ml2048_stream_wait")
        self._mirror_epoch = self._state_epoch
        return self._mirror

    def _mirror_field(self, views: dict[str, np.ndarray], key: str) -> np.ndarray:
        cur = self._cur
        if key == "state":
            return views["_board"][cur]
        if key == "valid_actions":
            return views["_valid"][cur]
        if key == "prev_state":
            return views["_board"][1 - cur]
        if key == "prev_valid_actions":
            return views["_valid"][1 - cur]
        if key == "terminated":
            return views["_terminated_padded"][: self._size]
        return views["_" + key]

    def _device_field(self, key: str, cur: Optional[int] = None) -> torch.Tensor:
        cur = self._cur if cur is None else cur
        if key == "state":
            return self._board[cur]
        if key == "valid_actions":
            return self._valid[cur]
        if key == "prev_state":
            return self._board[1 - cur]
        if key == "prev_valid_actions":
            return self._valid[1 - cur]
        if key == "merged":
            if self._merged is None:
                raise KeyError("merged is not tracked (track_merged=False)")
            return self._merged
        return {"step": self._step, "reward": self._reward, "score": self._score, "terminated": self._terminated,
                "invalid": self._invalid}[key]

    def _fetch(self, key: str, force_host: bool = False):
        t = self._device_field(key)
        if self._output == "torch" and not force_host:
            return t
        return self._to_host(t, key)

    def _upload_tables(self) -> None:
        """Tables changed on the host: ship the permutations (16 KiB) and fold the 2-vs-4 uniforms into
        a 16-bit mask (only randfloat[0:16] is ever read, indexed by CELL: game_numba.py:207)."""
        # Staged through a small ring of pinned buffers so that the upload (32 KiB, ~10 % of prepare() calls) is an
        # asynchronous copy: a pageable copy would make the host wait for everything queued on the stream.
        if self._tables_pin is None:
            self._tables_pin = torch.empty((4, 2, RAND_ROWS, 16), dtype=torch.uint8, pin_memory=True)
            self._tables_pin_np = self._tables_pin.numpy()
            self._tables_pin_events = [None] * 4
            self._tables_pin_next = 0
        k = self._tables_pin_next
        self._tables_pin_next = (k + 1) % 4
        if self._tables_pin_events[k] is not None:
            self._tables_pin_events[k].synchronize()  # the copy that last used this staging slot (4 refreshes ago)
        stage = self._tables_pin_np[k]
        stage[0] = self._randperm
        _lib.check(self._lib.ml2048_pack_randperm_keys(self._randperm.ctypes.data, stage[1].ctypes.data, RAND_ROWS),
                   "ml2048_pack_randperm_keys")
        self._table_slot = 0
        self._tables_dev[0].copy_(self._tables_pin[k], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self._tables_pin_events[k] = ev
        if self._rng_mode == _lib.RNG_REPLAY:  # Philox mode draws its epoch masks from the counter-based stream (_philox_epoch)
            self._two_mask = int(self._lib.ml2048_two_mask(self._randfloat.ctypes.data, self._two_prob))

    _TABLE_BYTES = 2 * RAND_ROWS * 16  # one slot of the table ring

    def _table_ptrs(self) -> tuple[int, int]:
        """(randperm, randperm_keys) device pointers of the slot eager calls use (slot 0 in scheduled mode:
        the kernels add entry.table * table_stride themselves)."""
        base = self._tables_dev.data_ptr() + (0 if self._sched_len else self._table_slot * self._TABLE_BYTES)
        return base, base + RAND_ROWS * 16

    # ------------------------------------------------------------------------------------------
    # device-resident schedule (CUDA-graph replay without host work)
    # ------------------------------------------------------------------------------------------

    def schedule_ahead(self, steps: int, *, min_steps: int = 1) -> int:
        """Pre-draw the host random numbers of the next ``steps`` runner steps (one prepare() + one step()
        each) and keep them on the device, so that prepare()/step() stop touching the host generator and a
        CUDA graph can replay them.  The draws are the reference's, in the reference's order
        (game_numba.py:622-626 then :670 per runner step); every table refresh inside the window takes one
        slot of the table ring.  Returns the number of steps scheduled.  ``steps = 0`` returns to eager mode."""
        if self._sched_len and self._sched_pos < self._sched_len:
            raise RuntimeError(f"{self._sched_len - self._sched_pos} scheduled steps are still pending")
        if steps <= 0:
            self._sched_len = self._sched_pos = 0
            self._upload_tables()
            return 0
        slots = max(int(min_steps) + 1, min(steps + 1, 64))
        if slots > self._table_slots:
            self._table_slots = slots
            self._tables_dev = torch.zeros((slots, 2, RAND_ROWS, 16), dtype=torch.uint8, device=self.device)
        ring = getattr(self, "_ring_host", None)
        if ring is None or ring.shape[0] < slots:
            ring = self._ring_host = np.zeros((slots, 2, RAND_ROWS, 16), dtype=np.uint8)

        def put(slot: int) -> None:
            ring[slot, 0] = self._randperm
            _lib.check(self._lib.ml2048_pack_randperm_keys(self._randperm.ctypes.data, ring[slot, 1].ctypes.data, RAND_ROWS),
                       "ml2048_pack_randperm_keys")
            if self._rng_mode == _lib.RNG_REPLAY:
                self._two_mask = int(self._lib.ml2048_two_mask(self._randfloat.ctypes.data, self._two_prob))

        put(0)  # the tables in force now
        slot = 0
        entries = np.zeros((steps, 4), dtype=np.int64)
        n = 0
        while n < steps and self._rng_mode != _lib.RNG_REPLAY:
            self._philox_epoch(self._philox_counter)  # Philox mode: the counter and the epoch's 2-vs-4 mask are the schedule
            entries[n, 2] = self._philox_counter
            entries[n, 3] = self._two_mask
            self._philox_counter += 2
            self._rand_step += 1
            n += 1
        while n < steps:
            coin = self._draw_coin()  # game_numba.py:622
            refresh = coin >= 0.9 or self._rand_step >= self._RAND_SIZE
            if refresh and slot + 1 >= slots:
                self._pending_coin = coin  # no ring slot left: this coin opens the next window
                break
            if refresh:
                self._rand_step = 0
                self._schedule.refresh_tables(self._randperm, self._randfloat)
                slot += 1
                put(slot)
            off_prepare = self._schedule.offset()
            off_step = self._schedule.offset()
            entries[n, 0] = self._rand_step + off_prepare
            entries[n, 1] = self._rand_step + off_step
            entries[n, 2] = self._philox_counter
            entries[n, 3] = self._two_mask | (slot << 32)
            self._philox_counter += 2
            self._rand_step += 1
            n += 1
        if n < min_steps:
            raise RuntimeError(f"could only schedule {n} < {min_steps} steps with {slots} table slots")
        self._tables_dev[: slot + 1].copy_(torch.from_numpy(ring[: slot + 1]))
        self._table_slot = slot  # where the tables in force at the end of the window live
        if self._sched_dev is None or self._sched_dev.shape[0] < steps:
            self._sched_dev = torch.zeros((steps, 4), dtype=torch.int64, device=self.device)  # fixed address from here on
        self._sched_dev[:n].copy_(torch.from_numpy(entries[:n]))
        self._sched_cursor_dev.zero_()
        self._sched_len, self._sched_pos = n, 0
        return n

    # ------------------------------------------------------------------------------------------
    # reference surface
    # ------------------------------------------------------------------------------------------

    def reset(self, seed: Optional[int] = None, *, schedule: Any = None) -> None:
        """game_numba.py:606-617.  ``schedule`` (optional) replaces the numpy generator by recorded draws."""
        self._schedule = schedule if schedule is not None else make_schedule(seed)
        self._sched_len = self._sched_pos = 0
        self._pending_coin = None
        self._rand_step = 0
        self._randperm[:, :] = np.arange(16).reshape((1, 16))
        self._schedule.refresh_tables(self._randperm, self._randfloat)
        self._upload_tables()
        self._philox_seed = int(seed) & 0xFFFFFFFFFFFFFFFF if seed is not None else int(np.random.SeedSequence().entropy) & 0xFFFFFFFFFFFFFFFF
        self._philox_counter = 0
        if self._rng_mode == _lib.RNG_PHILOX:
            self._philox_epoch(-1)  # the epoch in force after reset(): drawn at counter 2^64 - 1
        with torch.cuda.device(self.device):
            rc = self._lib.ml2048_reset_state(
                self._p(self._board[0]), self._p(self._board[1]), self._p(self._valid[0]), self._p(self._valid[1]),
                self._p(self._id), self._p(self._step), self._p(self._score), self._p(self._reward),
                self._p(self._terminated_padded), self._p(self._invalid), self._p(self._merged), self._size, self._stream())
        _lib.check(rc, "ml2048_reset_state")
        if self._onehot is not None:
            self._onehot.zero_()
            self._onehot[:, 0, :] = 1  # an all-empty board encodes as class 0 everywhere
        self._stats_dev.zero_()
        # the optional device logs restart with the environment: rows from before the reset must not mix with rows after it
        for name in ("_age", "_traj_state", "_traj_action", "_traj_score", "_traj_rows", "_ep_steps", "_ep_score", "_ep_max_tile"):
            t = getattr(self, name, None)
            if t is not None:
                t.zero_()
        self._cur = 0
        self._obs_cache = None
        self._state_epoch += 1
        self._id_bound = None  # upper bound of the id counter, re-read from the device on the next prepare()

    def observations(self):
        """game_numba.py:586-587: (board (M,16) u8, valid_actions (M,4) u8)."""
        cached = self._obs_cache
        if cached is not None:
            return cached
        return self._fetch("state"), self._fetch("valid_actions")

    def observations_onehot(self) -> torch.Tensor:
        """The fused CNN input, (M,16,16) class-major on the device (policy/_network.py:86-95)."""
        if self._onehot is None:
            raise RuntimeError("construct VecGame(..., onehot='f32'|'bf16'|'u8') to fuse the one-hot encoding")
        return self._onehot

    def afterstates(self, *, merged: bool = False) -> dict:
        """The four moves of every current board without the spawn (``ops.afterstates`` with this environment's
        ``reward_fn``): "state" (M,4,16), "reward" (M,4) -- what ``step(a)`` would return, 0 where the move does not change
        the board --, "valid_actions" (M,4) and, with ``merged=True``, "merged" (M,4,16).  CUDA tensors in torch mode, NumPy
        arrays (fresh copies) in NumPy mode.  Changes no state: boards, counters, schedule and host generator stay as they are."""
        from .ops import afterstates

        with self._guard:
            res = afterstates(self._board[self._cur], reward_fn=self._reward_fn, merged=merged)
        if self._output == "numpy":
            return {k: v.cpu().numpy() for k, v in res.items()}
        return res

    def prepare(self):
        """game_numba.py:619-658: refresh tables with probability 0.1, draw an offset, reset every
        terminated slot in ascending order.  Returns ``(indices,)``."""
        p = self._prep_args
        cur = self._cur
        self._state_epoch += 1
        self._check_id_range(1)
        if self._sched_len and self._sched_pos >= self._sched_len:
            self.schedule_ahead(self._sched_len)  # window used up: draw the next one (eager callers only)
        if self._sched_len:
            p.sched = self._sched_dev.data_ptr()
            p.sched_cursor = self._cursor_ptr[cur]
            p.table_stride = self._TABLE_BYTES
        else:
            p.sched = None
            p.rand_base, p.philox_counter = self._prepare_draws()
            p.two_mask = self._two_mask
        p.board = self._board_ptr[cur]
        p.valid = self._valid_ptr[cur]
        p.randperm = self._table_ptrs()[0]
        p.philox_seed = self._philox_seed
        stream = self._stream()
        with self._guard:
            if self._dist_group is None:
                _lib.check(self._lib.ml2048_prepare(C.byref(p), stream), "ml2048_prepare")
            else:
                self._prepare_sharded(p, stream)
        self._obs_cache = None
        if self._sync_free:
            return (None,)
        if self._output == "numpy" and self._size <= self._EAGER_HOST_MAX_GAMES:
            # count, index list and the post-reset observations behind one synchronisation
            views = self._mirror_to_host()
            self._obs_cache = (views["_board"][cur], views["_valid"][cur])
            return (views["_reset_indices_dev"][: int(views["_reset_count_dev"][0])].copy(),)
        if self._output == "numpy" and self._size <= self._BATCHED_HOST_MAX_GAMES:
            # the count and the post-reset observations behind one synchronisation; the index list only if non-empty
            cnt = self._pinned("_reset_count", self._reset_count_dev)
            cnt.copy_(self._reset_count_dev, non_blocking=True)
            got = self._fetch_many(("state", "valid_actions"))
            self._obs_cache = (got["state"], got["valid_actions"])
            n = int(cnt[0])
            return (self._reset_indices_dev[:n].cpu().numpy() if n else np.zeros((0,), dtype=np.int64),)
        if self._output == "numpy":
            # the count and a prefix of the index list that covers the steady state (1.6 % of the games; ~0.9 % finish per
            # step) behind ONE synchronisation, through pinned memory; the rest follows only if more games were over
            stage = getattr(self, "_idx_stage", None)
            if stage is None:
                cap = int(min(self._size, max(1 << 16, self._size >> 6)))
                stage = self._idx_stage = torch.empty((cap + 1,), dtype=torch.int64, pin_memory=True)
                self._idx_stage_np = stage.numpy()
            cap = stage.numel() - 1
            stream = self._stream()
            with self._guard:
                _lib.check(self._lib.ml2048_copy_async(stage.data_ptr(), self._reset_count_dev.data_ptr(), 8, stream), "ml2048_copy_async")
                _lib.check(self._lib.ml2048_copy_async(stage.data_ptr() + 8, self._reset_indices_dev.data_ptr(), 8 * cap, stream),
                           "ml2048_copy_async")
                _lib.check(self._lib.ml2048_stream_wait(stream), "ml2048_stream_wait")
            n = int(self._idx_stage_np[0])
            if n <= cap:
                return (self._idx_stage_np[1:1 + n].copy(),)
            return (self._reset_indices_dev[:n].cpu().numpy(),)
        n = int(self._reset_count_dev.item())
        return (self._reset_indices_dev[:n],)

    def _prepare_draws(self) -> tuple[int, int]:
        """The host half of one eager prepare() (game_numba.py:622-626): refresh the tables with probability 0.1, draw the
        row offset.  Returns (rand_base, the Philox counter this prepare uses)."""
        rand_offset = 0
        if self._rng_mode == _lib.RNG_REPLAY:  # Philox spawns need none of the reference's host draws
            if self._draw_coin() >= 0.9 or self._rand_step >= self._RAND_SIZE:
                self._rand_step = 0
                self._schedule.refresh_tables(self._randperm, self._randfloat)
                self._upload_tables()
            rand_offset = self._schedule.offset()
        else:
            self._philox_epoch(self._philox_counter)
        counter = self._philox_counter
        self._philox_counter += 1
        return self._rand_step + rand_offset, counter

    _COIN_REFRESH = int(0.9 * 4294967296.0)  # a 32-bit coin >= this value opens a new table epoch (game_numba.py:622)

    def _philox_epoch(self, counter: int) -> None:
        """Philox mode, host half of one prepare(): the reference's table-epoch logic (game_numba.py:622-624) with draws
        from the counter-based stream instead of the numpy generator.  The epoch's 16-bit mask ties the 2-vs-4 choice to
        the CELL, as the reference's ``randfloat[cell] < two_prob`` does (:207) -- that tie is part of the reference's
        episode statistics (tests: test_random_policy_episode_statistics_chi2_and_z)."""
        coin, mask = C.c_uint32(0), C.c_uint32(0)
        self._lib.ml2048_philox_epoch_draws(self._philox_seed, counter & 0xFFFFFFFFFFFFFFFF, self._two_prob, C.byref(coin), C.byref(mask))
        if coin.value >= self._COIN_REFRESH or self._rand_step >= self._RAND_SIZE or counter < 0:
            self._rand_step = 0
            self._two_mask = mask.value

    _ID_MAX = (1 << 31) - 1  # ids are int32 like the reference's `id` field (game_numba.py:538)

    def _check_id_range(self, prepares: int) -> None:
        """Game ids are int32 (the reference's record layout).  A prepare() hands out at most one id per game of the
        (global) batch, so the host keeps an UPPER BOUND of the device-resident id counter and raises before an id
        could wrap -- at 2^27 games and ~1 % resets per step that is after ~1700 steps.  The bound is refreshed from the
        device (one synchronisation) only when it comes within reach of 2^31, i.e. practically never for small batches."""
        if self._skip_id_check:
            return
        per_call = self._size * max(1, self._dist_world)
        bound = self._id_bound
        if bound is None or bound + prepares * per_call > self._ID_MAX:
            bound = int(self._game_count_dev.item())  # the true counter
            if bound + prepares * per_call > self._ID_MAX:
                # exact check is not possible without knowing how many games will end: refuse while a wrap is possible
                raise OverflowError(
                    f"game ids would pass int32: {bound} games started, up to {prepares * per_call} more in this call; "
                    "set env._game_count = 0 (ids restart) or use smaller shards")
        self._id_bound = bound + prepares * per_call

    def _draw_coin(self) -> float:
        coin = getattr(self, "_pending_coin", None)
        if coin is not None:
            self._pending_coin = None
            return coin
        return self._schedule.refresh_coin()

    def step(self, actions, *, fetch: Optional[tuple] = None, record: Optional[dict] = None) -> VecStepResult:
        """game_numba.py:660-698.  ``actions``: (M,) integers in 0..3 (NumPy array, CPU or CUDA tensor).

        ``record``: dict of CUDA tensors (one row of the caller's (use, step, game) rollout buffers, REPLAY_SPEC
        names and dtypes, replay.py:10-20) that the kernel fills with this transition -- what
        ``Trainer.on_stepped`` copies from the host in the reference (run_train3.py:138-149).

        ``fetch`` (NumPy mode, host actions): result keys the caller is going to read.  For large batches the
        step then runs as a pipeline over slices of the games -- actions H2D, kernel, results D2H on three
        streams -- so the PCIe copies in both directions overlap the kernel instead of following it."""
        assert tuple(actions.shape) == (self._size,), actions.shape  # game_numba.py:668
        if fetch and not record and self._can_pipeline(actions):
            return self._step_pipelined(actions, tuple(fetch))
        a = self._step_args
        host_actions = self._output == "numpy" and not self._sync_free and isinstance(actions, np.ndarray)
        eager_host = host_actions and self._size <= self._EAGER_HOST_MAX_GAMES
        batched_host = host_actions and not eager_host and self._size <= self._BATCHED_HOST_MAX_GAMES
        if eager_host or batched_host:
            dev_actions, a.action_dtype = self._stage_actions_pinned(actions)
        else:
            dev_actions, a.action_dtype = self._stage_actions(actions)
        a.action_mode = _lib.ACTIONS_GIVEN
        a.actions = dev_actions.data_ptr()
        a.actions_out = None
        self._set_record(record)
        self._launch_step()
        self._keepalive = dev_actions
        res = VecStepResult(self)
        if eager_host:
            # every field the reference's callers read (runner.py:165, replay.py:170-173, run_train3.py:138-149): one sync
            views = self._mirror_to_host()
            for k in VecStepResult.KEYS:
                if k != "merged" or self._merged is not None:
                    dict.__setitem__(res, k, self._mirror_field(views, k))
        elif batched_host:
            for k, v in self._fetch_many(self._COMMON_FIELDS).items():
                dict.__setitem__(res, k, v)  # merged / invalid stay lazy
        return res

    def _stage_actions_pinned(self, actions: np.ndarray) -> tuple[torch.Tensor, int]:
        """Host actions -> pinned staging -> asynchronous H2D (no pageable-copy synchronisation)."""
        if actions.dtype not in (np.int64, np.int32, np.uint8, np.int8):
            actions = actions.astype(np.int64)
        if actions.dtype == np.int8:
            actions = actions.view(np.uint8)
        tdtype = {np.dtype(np.int64): torch.int64, np.dtype(np.int32): torch.int32, np.dtype(np.uint8): torch.uint8}[actions.dtype]
        stage = self._host.get("_actions_stage")
        if stage is None or stage.dtype != tdtype:
            stage = torch.empty((self._size,), dtype=tdtype, pin_memory=True)
            self._host["_actions_stage"] = stage
            self._actions_stage_dev = torch.empty((self._size,), dtype=tdtype, device=self.device)
            self._host["_actions_stage_np"] = stage.numpy()
        self._host["_actions_stage_np"][...] = actions
        with self._guard:
            _lib.check(self._lib.ml2048_copy_async(self._actions_stage_dev.data_ptr(), stage.data_ptr(), stage.numel() * stage.element_size(),
                                                   self._stream()), "ml2048_copy_async")
        code = {torch.int64: _lib.ACT_I64, torch.int32: _lib.ACT_I32, torch.uint8: _lib.ACT_U8}[tdtype]
        return self._actions_stage_dev, code

    def step_from_logits(self, logits: torch.Tensor, *, log_prob_out: Optional[torch.Tensor] = None,
                         record: Optional[dict] = None) -> VecStepResult:
        """One step whose actions are SAMPLED INSIDE THE KERNEL from the policy head's logits (M,4) f32, masked by
        the current valid actions exactly like ``_sample_action`` (policy/actor_critic.py:56-76).  The sampled
        actions land in ``sampled_actions`` (uint8), their log-probabilities in ``log_prob_out`` (f32 (M,))."""
        if not (isinstance(logits, torch.Tensor) and logits.is_cuda and logits.dtype == torch.float32 and logits.is_contiguous()
                and tuple(logits.shape) == (self._size, 4)):
            raise ValueError(f"logits must be a contiguous CUDA float32 ({self._size},4) tensor")
        if log_prob_out is not None and not (log_prob_out.is_cuda and log_prob_out.dtype == torch.float32
                                             and log_prob_out.is_contiguous() and log_prob_out.numel() == self._size):
            raise ValueError("log_prob_out must be a contiguous CUDA float32 (M,) tensor")
        a = self._step_args
        a.action_mode = _lib.ACTIONS_FROM_LOGITS
        a.action_dtype = _lib.ACT_U8
        a.actions = None
        a.actions_out = self._p(self._actions_out)
        a.logits = logits.data_ptr()
        a.log_prob_out = self._p(log_prob_out)
        self._set_record(record)
        self._launch_step()
        a.logits = None
        a.log_prob_out = None
        self._keepalive = (logits, log_prob_out)
        return VecStepResult(self)

    @property
    def sampled_actions(self) -> torch.Tensor:
        """uint8 (M,): the actions the kernel chose in the last step_random(return_actions=True) / step_from_logits()."""
        return self._actions_out

    _RECORD_SPEC = {  # REPLAY_SPEC rows (replay.py:10-20) the step kernel can fill: name -> (trailing shape, dtypes)
        "state": ((16,), (torch.int8, torch.uint8)),
        "valid_actions": ((4,), (torch.bool, torch.uint8)),
        "action": ((), (torch.int8, torch.uint8)),
        "reward": ((), (torch.float32,)),
        "next_state": ((16,), (torch.int8, torch.uint8)),
        "next_valid_actions": ((4,), (torch.bool, torch.uint8)),
        "step": ((), (torch.int32,)),
        "terminated": ((), (torch.bool, torch.uint8)),
    }

    def _set_record(self, record: Optional[dict]) -> None:
        """Point the kernel's transition outputs at the caller's buffer rows (or clear them)."""
        a = self._step_args
        if not record and not self._record_active:
            return
        for name, (shape, dtypes) in self._RECORD_SPEC.items():
            t = record.get(name) if record else None
            if t is not None:
                if not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous() and t.dtype in dtypes
                        and tuple(t.shape) == (self._size,) + shape):
                    raise ValueError(f"record[{name!r}] must be a contiguous CUDA tensor {(self._size,) + shape} of {dtypes}")
            setattr(a, "tr_" + name, None if t is None else t.data_ptr())
        if record:
            unknown = set(record) - set(self._RECORD_SPEC)
            if unknown:
                raise KeyError(f"unknown record fields {sorted(unknown)}")
        self._record_active = bool(record)
        self._keep_record = record

    def summary(self) -> list[Any]:
        """game_numba.py:593-604: (tile value, count, share) of the max tile over all live boards."""
        hist = torch.zeros((20,), dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self._lib.ml2048_max_tile_hist(self._p(self._board[self._cur]), None, self._size, self._p(hist), self._stream())
        _lib.check(rc, "ml2048_max_tile_hist")
        counts = hist.cpu().numpy()
        total = counts.sum()
        entries = [(2 ** int(k), counts[k], counts[k] / total) for k in range(20) if counts[k]]
        entries.sort(key=lambda s: s[0], reverse=True)
        return entries

    @property
    def _data(self) -> _DataView:
        return _DataView(self)

    @property
    def _game_count(self) -> int:
        return int(self._game_count_dev.item())

    @_game_count.setter
    def _game_count(self, value: int) -> None:
        self._game_count_dev.fill_(int(value))
        self._id_bound = None

    @property
    def _prev_state(self):
        return self._fetch("prev_state")

    @property
    def _prev_valid_actions(self):
        return self._fetch("prev_valid_actions")

    # ------------------------------------------------------------------------------------------
    # extras: device-side policy for synthetic rollouts, statistics, sharding
    # ------------------------------------------------------------------------------------------

    def step_random(self, *, return_actions: bool = False, record: Optional[dict] = None, auto_reset: bool = False):
        """One step with uniformly random VALID actions chosen inside the kernel (Philox) --
        the benchmark policy (semantics of policy/random.py:17-27), no action array crosses the bus.

        ``auto_reset=True`` fuses the preceding ``prepare()`` into the same launch: the games that are over are reset
        first (slot-ordered ids, two tiles, the reference's draws in the reference's order) and then played.  Every
        array ends up exactly as after ``prepare(); step_random()`` -- including ``prev_state`` -- but the scattered
        writes of the reset ride on the step's coalesced ones and one launch (plus a 1-block-per-32k-games scan of the
        finished-game counts the previous step published) replaces two.  ``last_reset()`` returns what ``prepare()``
        would have returned."""
        a = self._step_args
        a.action_mode = _lib.ACTIONS_RANDOM_VALID
        a.action_dtype = _lib.ACT_U8
        a.actions = None
        a.actions_out = self._p(self._actions_out) if return_actions else None
        self._set_record(record)
        self._launch_step(fused_reset=auto_reset)
        return VecStepResult(self)

    def last_reset(self):
        """``(indices,)`` of the games the last prepare() / step_random(auto_reset=True) reset (synchronises)."""
        n = int(self._reset_count_dev.item())
        idx = self._reset_indices_dev[:n]
        return (idx if self._output == "torch" else idx.cpu().numpy(),)

    def _ensure_autoreset(self) -> None:
        """Buffers of the fused auto-reset (allocated on first use): the slot-ordered ranks of the finished games, which
        ml2048_autoreset_scan derives from the `terminated` flags right before a fused step."""
        if getattr(self, "_reset_rank", None) is not None:
            return
        groups = (self._size + 31) // 32
        chunks = (groups + 1023) // 1024
        dev = self.device
        self._reset_rank = torch.zeros((groups,), dtype=torch.int32, device=dev)
        self._reset_chunk_base = torch.zeros((chunks,), dtype=torch.int32, device=dev)
        self._reset_id_base = torch.zeros((1,), dtype=torch.int64, device=dev)
        self._ar_scratch = torch.zeros((int(self._lib.ml2048_autoreset_scratch_ints(self._size)),), dtype=torch.int32, device=dev)
        self._step_args.id = self._p(self._id)

    def _launch_autoreset_scan(self, stream: int) -> None:
        _lib.check(self._lib.ml2048_autoreset_scan(self._p(self._terminated_padded), self._reset_rank.data_ptr(),
                                                   self._reset_chunk_base.data_ptr(), self._size, self._p(self._game_count_dev), None,
                                                   self._reset_id_base.data_ptr(), self._p(self._reset_count_dev),
                                                   self._ar_scratch.data_ptr(), stream), "ml2048_autoreset_scan")

    def _launch_step(self, fused_reset: bool = False) -> None:
        a = self._step_args
        cur = self._cur
        self._obs_cache = None
        self._state_epoch += 1
        if fused_reset:
            if self._dist_group is not None:
                raise RuntimeError("auto_reset=True is not available with shard() (globally ordered ids need the per-rank counts "
                                   "between the scan and the step): call prepare() and step_random()")
            if self._record_active or self._step_args.episode_max_tile or self._step_args.traj_state:
                raise RuntimeError("auto_reset=True serves the lean kernels: no record=, episode log or trajectory log")
            self._ensure_autoreset()
            self._check_id_range(1)
            if self._sched_len and self._sched_pos >= self._sched_len:
                self.schedule_ahead(self._sched_len)
            a.reset_rank = self._reset_rank.data_ptr()
            a.reset_chunk_base = self._reset_chunk_base.data_ptr()
            a.reset_id_base = self._reset_id_base.data_ptr()
            a.reset_indices = self._p(self._reset_indices_dev)
            if not self._sched_len:
                a.rand_base, a.prepare_philox_counter = self._prepare_draws()  # prepare()'s host draws come first (:622-626)
        else:
            a.reset_rank = None
        if self._sched_len:
            if self._sched_pos >= self._sched_len:
                raise RuntimeError("the device schedule is used up: call prepare() (or schedule_ahead) first")
            a.sched = self._sched_dev.data_ptr()
            a.sched_cursor = self._cursor_ptr[cur]
            a.sched_cursor_next = self._cursor_ptr[1 - cur]
            a.table_stride = self._TABLE_BYTES
            self._sched_pos += 1
        else:
            rand_offset = self._schedule.offset() if self._rng_mode == _lib.RNG_REPLAY else 0  # game_numba.py:670
            a.sched = None
            a.rand_seed = self._rand_step + rand_offset  # :681
            self._rand_step += 1  # :685
            a.two_mask = self._two_mask
            a.philox_counter = self._philox_counter
            self._philox_counter += 1
        a.board_in = self._board_ptr[cur]
        a.board_out = self._board_ptr[1 - cur]
        a.valid_in = self._valid_ptr[cur]
        a.valid_out = self._valid_ptr[1 - cur]
        a.randperm, a.randperm_keys = self._table_ptrs()
        a.philox_seed = self._philox_seed
        stream = self._stream()
        with self._guard:
            if fused_reset:
                self._launch_autoreset_scan(stream)
            _lib.check(self._lib.ml2048_step(C.byref(a), stream), "ml2048_step")
        self._cur = 1 - cur

    # -- host-buffer pipeline -----------------------------------------------------------------------

    _PIPELINE_MIN_GAMES = 1 << 18
    # slices of the H2D / kernel / D2H pipeline: 8 at M >= 2^22, fewer below (0 = by batch size) -- a slice costs ~0.1 ms of
    # host time to enqueue, so slices of fewer than ~2^19 games make the HOST the bound (profiles/e2e_slices_r02.txt:
    # M = 2^18: 0.30 ms per step with one slice, 0.82 ms with eight; 2^20: 0.71 ms with two, 1.00 ms with eight)
    _PIPELINE_CHUNKS = int(os.environ.get("ML2048_PIPELINE_CHUNKS", "0"))
    _PIPELINE_MAX_CHUNKS = 8
    _PIPELINE_SLICE_GAMES = 1 << 19
    _PIPELINE_RAMP_MIN_GAMES = 1 << 23
    # slice sizes ramp up at the front (the D2H stream, which bounds this path, starts after a small slice's H2D + kernel
    # instead of a full-size one's) and down at the back (less left to expand on the host once the last copy has landed)
    _PIPELINE_RAMP = os.environ.get("ML2048_PIPELINE_RAMP", "1") != "0"
    # copy streams the slices alternate between (1, 2, 3 measured 7.35 / 7.41 / 7.42 ms per step at M = 2^24: the copies of one
    # stream already follow each other without a gap)
    _PIPELINE_D2H_STREAMS = int(os.environ.get("ML2048_D2H_STREAMS", "1"))
    _PACK_FLAGS = os.environ.get("ML2048_PACK_FLAGS", "1") != "0"  # one byte per game over PCIe for mask + terminated + invalid
    # host threads that expand a slice of packed flags: a share of the host's cores (one process per GPU shares them)
    _UNPACK_THREADS = int(os.environ.get("ML2048_UNPACK_THREADS", "0")) or max(
        1, min(4, (os.cpu_count() or 4) // (2 * max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1"))))))  # (2-4 measured best; more only contend)

    def _can_pipeline(self, actions) -> bool:
        if self._output != "numpy" or self._sched_len or self._size < self._PIPELINE_MIN_GAMES:
            return False
        if isinstance(actions, np.ndarray):
            return actions.dtype in (np.int64, np.int32, np.uint8, np.int8)
        return isinstance(actions, torch.Tensor) and actions.device.type == "cpu" and actions.dtype in (
            torch.int64, torch.int32, torch.uint8, torch.int8)

    def _pipeline_bounds(self, m: int) -> list[int]:
        """Slice boundaries of the pipelined step (multiples of 256 games, strictly increasing, 0 .. m)."""
        got = getattr(self, "_pipe_bounds", None)
        if got is not None and got[-1] == m:
            return got
        chunks = self._PIPELINE_CHUNKS or min(self._PIPELINE_MAX_CHUNKS, max(1, -(-m // self._PIPELINE_SLICE_GAMES)))
        if self._PIPELINE_RAMP and chunks >= 4 and m >= self._PIPELINE_RAMP_MIN_GAMES:
            weights = [1, 2, 4] + [8] * (chunks - 2) + [4, 2, 1]
        else:
            weights = [1] * chunks
        total, acc, bounds = sum(weights), 0, [0]
        for w in weights[:-1]:
            acc += w
            b = min(m, (m * acc // total + 255) // 256 * 256)
            if b > bounds[-1]:
                bounds.append(b)
        if bounds[-1] < m:
            bounds.append(m)
        self._pipe_bounds = bounds
        return bounds

    def _step_pipelined(self, actions, fetch: tuple) -> VecStepResult:
        if isinstance(actions, np.ndarray):
            actions = torch.from_numpy(np.ascontiguousarray(actions))
        actions = actions.contiguous()
        code = {torch.int64: _lib.ACT_I64, torch.int32: _lib.ACT_I32, torch.uint8: _lib.ACT_U8, torch.int8: _lib.ACT_U8}[actions.dtype]
        m = self._size
        if getattr(self, "_pipe_streams", None) is None:
            self._pipe_streams = (torch.cuda.Stream(device=self.device),
                                  [torch.cuda.Stream(device=self.device) for _ in range(max(1, self._PIPELINE_D2H_STREAMS))])
            self._pipe_actions = {}
        h2d, d2h_streams = self._pipe_streams
        dev_actions = self._pipe_actions.get(actions.dtype)
        if dev_actions is None:
            dev_actions = torch.empty((m,), dtype=actions.dtype, device=self.device)
            self._pipe_actions[actions.dtype] = dev_actions
        main = torch.cuda.current_stream(self.device)
        cur = self._cur
        # this path launches by itself (not through _launch_step): drop what that would have dropped -- the cached
        # observations of prepare() and the transition-record pointers of an earlier step(record=...), which a
        # chunked launch must not write through
        self._obs_cache = None
        self._set_record(None)
        self._state_epoch += 1
        # the host draws of this step, once (game_numba.py:670, :681, :685)
        rand_offset = self._schedule.offset() if self._rng_mode == _lib.RNG_REPLAY else 0
        rand_seed = self._rand_step + rand_offset
        self._rand_step += 1
        counter = self._philox_counter
        self._philox_counter += 1
        fields = {k: self._device_field(k, 1 - cur) for k in fetch}  # the post-step buffers
        host = {}
        for k, t in fields.items():
            buf = self._host.get(k)
            if buf is None or buf.shape != t.shape or buf.dtype != t.dtype:
                buf = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
                self._host[k] = buf
            host[k] = buf
        # valid_actions (4 bytes), terminated and invalid cross PCIe as ONE byte per game (ml2048_pack_flags on the device,
        # ml2048_unpack_flags on the host, slice by slice while the later slices are still in flight): the D2H stream is what
        # bounds this path, and the three arrays are 6 of the 26 bytes a game's full result takes
        # (only when the 4-byte mask is wanted: terminated / invalid alone are a byte each already)
        flag_keys = [k for k in ("valid_actions", "terminated", "invalid") if k in fields] if self._PACK_FLAGS and "valid_actions" in fields else []
        packed_dev = packed_host = None
        if flag_keys:
            packed_dev = getattr(self, "_pipe_packed", None)
            if packed_dev is None:
                packed_dev = self._pipe_packed = torch.empty((m,), dtype=torch.uint8, device=self.device)
                self._pipe_packed_host = torch.empty((m,), dtype=torch.uint8, pin_memory=True)
            packed_host = self._pipe_packed_host
        slices = []
        a = _lib.StepArgs.from_buffer_copy(self._step_args)
        a.action_mode, a.action_dtype, a.actions_out, a.sched = _lib.ACTIONS_GIVEN, code, None, None
        a.reset_rank = None  # (left over from an earlier step_random(auto_reset=True))
        a.rand_seed, a.two_mask, a.philox_counter, a.philox_seed = rand_seed, self._two_mask, counter, self._philox_seed
        a.randperm_keys = self._table_ptrs()[1]
        esz = actions.element_size()
        bounds = self._pipeline_bounds(m)
        h2d.wait_stream(main)
        for d2h in d2h_streams:
            d2h.wait_stream(main)
        raw_main = main.cuda_stream
        # tools/e2e_timeline.py: when a list is hung here, every slice appends (lo, hi, event after its kernels, event after its copies)
        trace = getattr(self, "_pipe_trace", None)
        if trace is not None:
            ev_start = torch.cuda.Event(enable_timing=True)
            ev_start.record(main)
            trace.append((0, 0, ev_start, ev_start))
        with self._guard:
            for i, (lo, hi) in enumerate(zip(bounds[:-1], bounds[1:])):
                d2h = d2h_streams[i % len(d2h_streams)]  # slices alternate between the copy streams: no gap between their copies
                with torch.cuda.stream(h2d):
                    dev_actions[lo:hi].copy_(actions[lo:hi], non_blocking=True)
                main.wait_stream(h2d)
                a.num_games = hi - lo
                a.slot_base = self._slot_base + lo
                a.board_in = self._board_ptr[cur] + 16 * lo
                a.board_out = self._board_ptr[1 - cur] + 16 * lo
                a.valid_in = self._valid_ptr[cur] + 4 * lo
                a.valid_out = self._valid_ptr[1 - cur] + 4 * lo
                a.actions = dev_actions.data_ptr() + esz * lo
                a.step = self._step.data_ptr() + 8 * lo   # {step, score} records
                a.score = self._score.data_ptr() + 8 * lo
                a.reward = self._reward.data_ptr() + 4 * lo
                a.terminated = self._terminated_padded.data_ptr() + lo
                a.invalid = self._invalid.data_ptr() + lo
                a.merged = None if self._merged is None else self._merged.data_ptr() + 16 * lo
                if self._onehot is not None:
                    a.onehot_out = self._onehot.data_ptr() + lo * 256 * self._onehot.element_size()
                if self._step_args.id:
                    a.id = self._id.data_ptr() + 4 * lo
                if self._step_args.age:
                    a.age = self._age.data_ptr() + 4 * lo
                _lib.check(self._lib.ml2048_step(C.byref(a), raw_main), "ml2048_step")
                if flag_keys:
                    _lib.check(self._lib.ml2048_pack_flags(
                        a.valid_out, a.terminated if "terminated" in fields else None, a.invalid if "invalid" in fields else None,
                        packed_dev.data_ptr() + lo, hi - lo, raw_main), "ml2048_pack_flags")
                if trace is not None:
                    ev_kernel = torch.cuda.Event(enable_timing=True)
                    ev_kernel.record(main)
                d2h.wait_stream(main)
                with torch.cuda.stream(d2h):
                    if flag_keys:
                        packed_host[lo:hi].copy_(packed_dev[lo:hi], non_blocking=True)
                        done = torch.cuda.Event()
                        done.record(d2h)
                        slices.append((lo, hi, done))
                    for k, t in fields.items():
                        if k not in flag_keys:
                            host[k][lo:hi].copy_(t[lo:hi], non_blocking=True)
                    if trace is not None:
                        ev_copied = torch.cuda.Event(enable_timing=True)
                        ev_copied.record(d2h)
                        trace.append((lo, hi, ev_kernel, ev_copied))
        self._cur = 1 - cur  # only now: an exception above leaves the ping-pong state where it was
        # bytes this call moves over PCIe towards the host (for callers that account for them: bench.py's e2e)
        self.last_step_d2h_bytes = sum(t.numel() * t.element_size() for k, t in fields.items() if k not in flag_keys) + (m if flag_keys else 0)
        if flag_keys:
            ptr = {k: (host[k].data_ptr() if k in fields else None) for k in ("valid_actions", "terminated", "invalid")}
            n = len(slices)
            lo_arr = (C.c_int64 * n)(*[sl[0] for sl in slices])
            hi_arr = (C.c_int64 * n)(*[sl[1] for sl in slices])
            ev_arr = (C.c_void_p * n)(*[sl[2].cuda_event for sl in slices])
            # one call: the library's worker threads wait for each slice's event themselves and expand it while the slices
            # behind it are still in flight
            _lib.check(self._lib.ml2048_unpack_flags_sliced(packed_host.data_ptr(), n, lo_arr, hi_arr, ev_arr, ptr["valid_actions"],
                                                            ptr["terminated"], ptr["invalid"], self._UNPACK_THREADS), "ml2048_unpack_flags_sliced")
        for d2h in d2h_streams:
            d2h.synchronize()
        res = VecStepResult(self)
        for k in fetch:
            dict.__setitem__(res, k, host[k].numpy())
        return res

    def _stage_actions(self, actions) -> tuple[torch.Tensor, int]:
        if isinstance(actions, np.ndarray):
            if actions.dtype not in (np.int64, np.int32, np.uint8, np.int8):
                actions = actions.astype(np.int64)
            actions = torch.from_numpy(np.ascontiguousarray(actions))
        if not isinstance(actions, torch.Tensor):
            raise TypeError(f"actions must be a numpy array or torch tensor, got {type(actions)}")
        if actions.dtype not in (torch.int64, torch.int32, torch.uint8, torch.int8):
            actions = actions.to(torch.int64)
        if actions.device != self.device:
            actions = actions.to(self.device, non_blocking=True)
        actions = actions.contiguous()
        code = {torch.int64: _lib.ACT_I64, torch.int32: _lib.ACT_I32, torch.uint8: _lib.ACT_U8, torch.int8: _lib.ACT_U8}
        return actions, code[actions.dtype]

    def configure(self, *, output: Optional[str] = None, sync_free: Optional[bool] = None) -> None:
        """Switch between host (NumPy) and device (torch) results, or the sync-free prepare(), on a live environment."""
        if output is not None:
            if output not in ("numpy", "torch"):
                raise ValueError(f"output={output!r}")
            self._output = output
        if sync_free is not None:
            self._sync_free = bool(sync_free)

    def state_dict(self) -> dict[str, Any]:
        """Snapshot of the whole environment (device tensors are cloned, host random schedule copied).
        The reference never checkpoints the environment (SURVEY.md section 5); this makes rollouts
        restartable and lets a benchmark replay a recorded trajectory."""
        import copy

        if self._sched_len:
            raise RuntimeError("state_dict() while a device schedule is active is not supported: call schedule_ahead(0) first")
        torch.cuda.current_stream(self.device).synchronize()
        tensors = {
            name: getattr(self, name).clone()
            for name in ("_board", "_valid", "_id", "_step_score", "_reward", "_terminated_padded", "_invalid",
                         "_tables_dev", "_game_count_dev", "_stats_dev")
        }
        if self._merged is not None:
            tensors["_merged"] = self._merged.clone()
        if self._onehot is not None:
            tensors["_onehot"] = self._onehot.clone()
        # the optional device logs (enable_episode_log / enable_trajectory_log) belong to the state: a restored
        # environment continues its rows where the snapshot left them
        for name in ("_age", "_traj_state", "_traj_action", "_traj_score", "_traj_rows", "_ep_steps", "_ep_score", "_ep_max_tile"):
            t = getattr(self, name, None)
            if t is not None:
                tensors[name] = t.clone()
        host = {
            "size": self._size,
            "cur": self._cur,
            "rand_step": self._rand_step,
            "randperm": self._randperm.copy(),
            "randfloat": self._randfloat.copy(),
            "two_mask": self._two_mask,
            "philox_seed": self._philox_seed,
            "philox_counter": self._philox_counter,
            "schedule": copy.deepcopy(self._schedule),
            "table_slot": self._table_slot,
            "pending_coin": getattr(self, "_pending_coin", None),
        }
        return {"tensors": tensors, "host": host}

    def load_state_dict(self, sd: dict[str, Any]) -> None:
        import copy

        host = sd["host"]
        if host["size"] != self._size:
            raise ValueError(f"snapshot holds {host['size']} games, this environment {self._size}")
        for name, t in sd["tensors"].items():
            dst = getattr(self, name, None)
            if dst is None:
                raise ValueError(f"snapshot has {name} but this environment does not track it")
            if name != "_tables_dev" and dst.shape != t.shape:
                raise ValueError(f"snapshot {name} has shape {tuple(t.shape)}, this environment {tuple(dst.shape)}")
            if name == "_tables_dev" and dst.shape != t.shape:
                self._tables_dev = t.clone()
                self._table_slots = t.shape[0]
                continue
            dst.copy_(t)
        self._cur = host["cur"]
        self._rand_step = host["rand_step"]
        self._randperm[...] = host["randperm"]
        self._randfloat[...] = host["randfloat"]
        self._two_mask = host["two_mask"]
        self._philox_seed = host["philox_seed"]
        self._philox_counter = host["philox_counter"]
        self._schedule = copy.deepcopy(host["schedule"])
        self._table_slot = host.get("table_slot", 0)
        self._pending_coin = host.get("pending_coin")
        self._sched_len = self._sched_pos = 0
        self._obs_cache = None
        self._state_epoch += 1
        self._id_bound = None

    def enable_episode_log(self, capacity: int, id_base: int = 0) -> None:
        """Record (steps, score, max tile) of every finished game whose id lies in [id_base, id_base+capacity),
        indexed by id -- the statistic eval_perf.py collects for the games with ``id < rounds``
        (eval_perf.py:80-102) -- inside the step kernel, with no per-step host work."""
        if capacity <= 0:
            raise ValueError(f"capacity={capacity}")
        dev = self.device
        self._ep_steps = torch.zeros((capacity,), dtype=torch.int32, device=dev)
        self._ep_score = torch.zeros((capacity,), dtype=torch.float32, device=dev)
        self._ep_max_tile = torch.zeros((capacity,), dtype=torch.uint8, device=dev)
        a = self._step_args
        a.id = self._p(self._id)
        a.episode_id_base = int(id_base)
        a.episode_capacity = int(capacity)
        a.episode_steps = self._p(self._ep_steps)
        a.episode_score = self._p(self._ep_score)
        a.episode_max_tile = self._p(self._ep_max_tile)

    def enable_trajectory_log(self, capacity: int, max_rows: int = 4096, id_base: int = 0) -> None:
        """Capture whole episodes of the games with id in [id_base, id_base+capacity) on the device: one row
        (prev_state, action, score) per runner step plus the final (state, 0, score) row, like ``ReplayRecorder``
        (replay.py:161-201) but inside the step kernel.  ``max_rows`` bounds the rows kept per game."""
        if capacity <= 0 or max_rows <= 1:
            raise ValueError((capacity, max_rows))
        dev = self.device
        self._age = torch.zeros((self._size,), dtype=torch.int32, device=dev)
        self._traj_state = torch.zeros((capacity, max_rows, 16), dtype=torch.int8, device=dev)
        self._traj_action = torch.zeros((capacity, max_rows), dtype=torch.int8, device=dev)
        self._traj_score = torch.zeros((capacity, max_rows), dtype=torch.float32, device=dev)
        self._traj_rows = torch.zeros((capacity,), dtype=torch.int32, device=dev)
        a = self._step_args
        a.id = self._p(self._id)
        a.age = self._p(self._age)
        a.traj_id_base, a.traj_capacity, a.traj_max_rows = int(id_base), int(capacity), int(max_rows)
        a.traj_state = self._p(self._traj_state)
        a.traj_action = self._p(self._traj_action)
        a.traj_score = self._p(self._traj_score)
        a.traj_rows = self._p(self._traj_rows)
        self._prep_args.age = self._p(self._age)

    def trajectory(self, index: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """(state (rows,16) int8, action (rows,) int8, score (rows,) f32) of game id ``id_base + index`` so far --
        ``RecordBuffer.contiguous_result()`` (replay.py:86-107): rows = steps + 1 once the game is over."""
        if getattr(self, "_traj_rows", None) is None:
            raise RuntimeError("call enable_trajectory_log(capacity) first")
        rows = int(self._traj_rows[index].item())
        return self._traj_state[index, :rows], self._traj_action[index, :rows], self._traj_score[index, :rows]

    def episode_log(self) -> dict[str, torch.Tensor]:
        """Device tensors indexed by (game id - id_base): ``steps`` i32, ``score`` f32, ``max_tile`` u8 (0 = unfinished)."""
        if getattr(self, "_ep_max_tile", None) is None:
            raise RuntimeError("call enable_episode_log(capacity) first")
        return {"steps": self._ep_steps, "score": self._ep_score, "max_tile": self._ep_max_tile}

    def episode_stats(self, *, reset: bool = False) -> dict[str, Any]:
        """Finished-episode statistics accumulated by step(): RunnerStats' max-tile histogram
        (runner.py:150-166) plus episode count, score and step sums, max score."""
        raw = self.episode_stats_tensor()
        if reset:
            self._stats_dev.zero_()
        return stats_to_dict(raw.cpu())

    def episode_stats_tensor(self) -> torch.Tensor:
        """int64[24] on the device: hist[20], episodes, score_sum, step_sum, score_max (replicas folded)."""
        s = self._stats_dev
        return torch.cat([s[:, :23].sum(dim=0), s[:, 23:].max(dim=0).values])

    def shard(self, group: Any = None) -> None:
        """Make game ids globally slot-ordered across the ranks of ``group`` (each rank owning the
        contiguous global slots [slot_base, slot_base+size)), as in a single-process reference run:
        prepare() then exchanges per-rank reset counts (one tiny all_gather, no host sync)."""
        import torch.distributed as dist

        self._dist_group = group if group is not None else dist.group.WORLD
        self._dist_rank = dist.get_rank(self._dist_group)
        self._dist_world = dist.get_world_size(self._dist_group)
        self._counts_all = torch.zeros((self._dist_world,), dtype=torch.int64, device=self.device)

    def _prepare_sharded(self, p: Any, stream: int) -> None:
        import torch.distributed as dist

        p.id_offset = self._p(self._id_offset_dev)
        _lib.check(self._lib.ml2048_prepare_count(C.byref(p), stream), "ml2048_prepare_count")
        dist.all_gather_into_tensor(self._counts_all, self._reset_count_dev, group=self._dist_group)
        self._id_offset_dev.copy_(self._counts_all[: self._dist_rank].sum().reshape(1))
        _lib.check(self._lib.ml2048_prepare_apply(C.byref(p), stream), "ml2048_prepare_apply")
        self._game_count_dev += self._counts_all.sum()


def stats_to_dict(raw: torch.Tensor) -> dict[str, Any]:
    raw = raw.to(torch.int64).cpu().numpy()
    episodes = int(raw[20])
    return {
        "max_tile_hist": raw[:20].copy(),
        "episodes": episodes,
        "score_sum": int(raw[21]),
        "step_sum": int(raw[22]),
        "score_max": int(raw[23]),
        "mean_score": (int(raw[21]) / episodes) if episodes else float("nan"),
        "mean_steps": (int(raw[22]) / episodes) if episodes else float("nan"),
    }
