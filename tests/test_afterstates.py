"""
Afterstates (``ops.afterstates``, ``VecGame.afterstates``, ``ml2048_afterstates``): the four moves of every board without the
spawn.  Bit-exact against the live reference's board set, the reference's own line table, the C oracle and the
environment's own step.  The argument checks run without a GPU.

- Golden [GPU]: ``boards.npz`` for all four reward kinds with ``merged``: afterstate, ``merged``, mask, and the f32 reward cast
  to f64 ``==`` the fixture.
- Every line [GPU]: all 18^4 lines as each row and each column, noise in the other cells (exponents 16 and 17 included),
  against ``pushed_first`` / ``pushed_last``; where only that line can move, the mask against ``movable_*``, the normal reward
  and ``merged`` against the table's fusions.
- The environment's own step [GPU]: a ``VecGame`` at M = 70 001 after 50 random steps (four reward kinds in replay mode,
  ``improved`` in Philox mode), ``step(full a)`` from one snapshot for every a.  A valid move's stepped board equals the
  afterstate except in one cell (0 there, 1 or 2 after the step), with the same reward (bitwise) and ``merged``; an invalid
  one leaves the board, and the afterstate has reward 0 and empty ``merged``; ``valid_actions == 1 - invalid``.
  ``VecGame.afterstates()`` in torch and NumPy mode equals the op and leaves ``state_dict()``, the state epoch and the host
  generator as they were.
- Sizes [GPU]: M = 1, 3, 255, 256, 257, 2^20 + 3 (uint8 and int8 boards, with and without ``merged``) against the C oracle
  with canary bytes around every output; M = 2^24: tile sums conserved, normal reward = sum_k merged[k] * 2^(k+1), mask =
  ``ops.valid_actions``, 65 536 seeded rows against the oracle; M = 2^25 + 1, where the afterstate's byte offset passes 2^31,
  with a 2 GiB guard before that buffer (a wrapped offset lands in it).
- CUDA graph [GPU]: ``ops.afterstates(static_board, out=static_out)`` replayed on new boards equals eager calls.
- Errors: the C entry's -1 / -2 / -3 / -4 before any launch and the Python ``ValueError``s without a GPU; ``out`` entries of
  the wrong shape, dtype, device or layout on the GPU.
"""

from __future__ import annotations

import numpy as np
import pytest
import torch

from conftest import golden

KINDS = ("normal", "improved", "rank", "maxcell")
CANARY = 0xA5
KEYS = ("state", "reward", "valid_actions", "merged")
SHAPES = {"state": ((4, 16), torch.uint8), "reward": ((4,), torch.float32), "valid_actions": ((4,), torch.uint8),
          "merged": ((4, 16), torch.uint8)}


@pytest.fixture(scope="module")
def lib():
    from ml2048_b200 import _lib, build

    build.build()  # nvcc cross-compiles without a GPU; no-op when up to date
    return _lib.load()


@pytest.fixture(scope="module")
def ops(lib):
    from ml2048_b200 import ops

    return ops


def _gpu():
    assert torch.cuda.is_available()
    return torch.device("cuda")


def _random_boards(m: int, seed: int) -> np.ndarray:
    """Boards with exponents 0..15 (no out-of-domain fusions: the oracle logs only exponents below 16): an eighth from 0..3
    (many fusions per move), an eighth without empty cells (few valid directions, dead boards), every 97th of the rest empty,
    the rest with about 40 % empty cells."""
    rng = np.random.default_rng(seed)
    u = np.arange(256)
    wide = np.where(u < 102, 0, u % 15 + 1).astype(np.uint8)      # 40 % empty, else 1..15
    narrow = np.where(u < 64, 0, u % 3 + 1).astype(np.uint8)      # 25 % empty, else 1..3: many fusions per move
    b = wide[rng.integers(0, 256, size=(m, 16), dtype=np.uint8)]
    full = (u % 15 + 1).astype(np.uint8)                          # no empty cell: few valid directions, dead boards
    k = m // 8
    b[:k] = narrow[rng.integers(0, 256, size=(k, 16), dtype=np.uint8)]
    b[k:2 * k] = full[rng.integers(0, 256, size=(k, 16), dtype=np.uint8)]
    b[2 * k::97] = 0
    return b


def _oracle_rows(oracle, boards: np.ndarray, kind: str):
    """(after, reward f64, valid, merged) of every row from the C oracle, one board and one direction at a time."""
    n = boards.shape[0]
    after = np.empty((n, 4, 16), np.uint8)
    merged = np.empty((n, 4, 16), np.uint8)
    reward = np.empty((n, 4), np.float64)
    valid = np.empty((n, 4), np.uint8)
    for i in range(n):
        b = boards[i]
        for a in range(4):
            nb, mg = oracle.board_move(b, a)
            moved = bool((nb != b).any())
            after[i, a], merged[i, a], valid[i, a] = nb, mg, moved
            reward[i, a] = oracle.board_reward(kind, nb, b, mg) if moved else 0.0
    return after, reward, valid, merged


def _check_rows(oracle, boards: np.ndarray, res: dict, rows: np.ndarray, kind: str) -> None:
    after, reward, valid, merged = _oracle_rows(oracle, boards[rows], kind)
    np.testing.assert_array_equal(res["state"][rows], after)
    np.testing.assert_array_equal(res["valid_actions"][rows], valid)
    np.testing.assert_array_equal(res["reward"][rows].astype(np.float64), reward)
    if "merged" in res:
        np.testing.assert_array_equal(res["merged"][rows], merged)


def _guarded_out(m: int, merged: bool, dev, pad: int = 256, lead: dict | None = None):
    """Output tensors carved out of canary-filled buffers: `pad` bytes (or lead[key]) before and `pad` after each."""
    out, raw = {}, {}
    for k in KEYS if merged else KEYS[:3]:
        shape, dtype = SHAPES[k]
        nbytes = m * int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        before = (lead or {}).get(k, pad)
        buf = torch.full((before + nbytes + pad,), CANARY, dtype=torch.uint8, device=dev)
        out[k] = buf[before:before + nbytes].view(dtype).view((m,) + shape)
        raw[k] = (buf, before, nbytes)
    return out, raw


def _canaries_intact(raw) -> None:
    for k, (buf, before, nbytes) in raw.items():
        head, tail = bool((buf[:before] == CANARY).all()), bool((buf[before + nbytes:] == CANARY).all())
        assert head, f"{k}: bytes before the buffer were written"
        assert tail, f"{k}: bytes after the buffer were written"


def _host(res: dict) -> dict:
    return {k: v.cpu().numpy() for k, v in res.items()}


# ---------------------------------------------------------------------------------------------
# golden fixtures from the live reference
# ---------------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_golden_board_set(ops, kind):
    """The reference-generated board set (exponents up to 15, dead and empty boards): every direction, every reward kind."""
    g = golden("boards.npz")
    j = [str(x) for x in g["reward_names"]].index(kind)
    res = _host(ops.afterstates(torch.from_numpy(g["boards"]).to(_gpu()), reward_fn=kind, merged=True))
    np.testing.assert_array_equal(res["state"], g["moved"])
    np.testing.assert_array_equal(res["merged"], g["merged"])
    np.testing.assert_array_equal(res["valid_actions"], g["mask"])
    np.testing.assert_array_equal(res["reward"].astype(np.float64), g["rewards"][..., j])


@pytest.mark.gpu
def test_every_line_every_position_every_direction(ops):
    """All 18^4 lines as each row (left/right) and each column (up/down), noise in the other cells (exponents 16 and 17
    included), against the reference's _push_row table; on boards where only that line can move, the mask against
    _line_movable and the normal reward and `merged` against the table's fusions."""
    tab = golden("line_table.npz")
    v = np.arange(18, dtype=np.uint8)
    lines = np.stack(np.meshgrid(v, v, v, v, indexing="ij"), axis=-1).reshape(-1, 4)
    n = lines.shape[0]
    rng = np.random.default_rng(1)
    weights = (2 << np.arange(18)).astype(np.int64)
    dev = _gpu()
    for axis, dirs in (("row", (0, 1)), ("col", (2, 3))):
        for pos in range(4):
            boards = rng.integers(0, 18, size=(n, 16)).astype(np.uint8).reshape(n, 4, 4)
            if axis == "row":
                boards[:, pos, :] = lines
            else:
                boards[:, :, pos] = lines
            res = _host(ops.afterstates(torch.from_numpy(boards.reshape(n, 16)).to(dev)))
            for a in dirs:
                pushed = tab["pushed_first" if a in (0, 2) else "pushed_last"]
                out = res["state"][:, a].reshape(n, 4, 4)
                got = out[:, pos, :] if axis == "row" else out[:, :, pos]
                bad = np.flatnonzero((got != pushed).any(axis=1))
                assert bad.size == 0, (a, pos, lines[bad[0]], got[bad[0]], pushed[bad[0]])
        filler = np.array([[1, 2, 3, 4], [5, 6, 7, 8], [9, 10, 11, 12], [13, 14, 15, 16]], np.uint8)
        boards = np.broadcast_to(filler if axis == "row" else filler.T, (n, 4, 4)).copy()
        if axis == "row":
            boards[:, 0, :] = lines
        else:
            boards[:, :, 0] = lines
        res = _host(ops.afterstates(torch.from_numpy(boards.reshape(n, 16)).to(dev), merged=True))
        for a in dirs:
            name = "first" if a in (0, 2) else "last"
            fused = tab[f"fused_{name}"]
            np.testing.assert_array_equal(res["valid_actions"][:, a], tab[f"movable_{name}"].astype(np.uint8))
            want_gain = np.where(fused > 0, weights[fused], 0).sum(axis=1)
            np.testing.assert_array_equal(res["reward"][:, a].astype(np.int64), want_gain)
            want_merged = np.zeros((n, 18), np.uint8)
            for j in range(2):
                np.add.at(want_merged, (np.arange(n), fused[:, j]), (fused[:, j] > 0).astype(np.uint8))
            np.testing.assert_array_equal(res["merged"][:, a], want_merged[:, :16])  # exponents 16, 17 have no slot


# ---------------------------------------------------------------------------------------------
# against the environment's own step
# ---------------------------------------------------------------------------------------------


def _played_env(kind: str, rng_mode: str, m: int = 70001, steps: int = 50):
    import ml2048_b200

    env = ml2048_b200.VecGame(m, kind, output="torch", rng_mode=rng_mode)
    env.reset(1234)
    rng = np.random.default_rng(99)
    for _ in range(steps):
        env.prepare()
        env.step(torch.from_numpy(rng.integers(0, 4, size=m)).to(env.device))
    env.prepare()
    return env


@pytest.mark.gpu
@pytest.mark.parametrize("kind,rng_mode", [(k, "replay") for k in KINDS] + [("improved", "philox")])
def test_against_the_environments_step(ops, kind, rng_mode):
    """After 50 random steps: step(a) for every a from the same snapshot equals the afterstate plus one spawned tile where
    the move was valid (same reward bit for bit, same `merged`), and leaves the board alone where it was not."""
    env = _played_env(kind, rng_mode)
    m = env._size
    board = env._board[env._cur].clone()
    res = ops.afterstates(board, reward_fn=kind, merged=True)
    sd = env.state_dict()
    for a in range(4):
        r = env.step(torch.full((m,), a, dtype=torch.int64, device=env.device))
        valid = res["valid_actions"][:, a]
        assert torch.equal(valid, 1 - r["invalid"]), a
        mv = valid.bool()
        assert 0 < int(mv.sum()) < m  # both kinds of games are present
        after, stepped = res["state"][:, a][mv], r["state"][mv]
        diff = after != stepped
        assert bool((diff.sum(dim=1) == 1).all()), a
        assert bool((after[diff] == 0).all()) and bool(((stepped[diff] == 1) | (stepped[diff] == 2)).all()), a
        assert torch.equal(res["reward"][:, a][mv].view(torch.int32), r["reward"][mv].view(torch.int32)), a
        assert torch.equal(res["merged"][:, a][mv], r["merged"][mv]), a
        assert torch.equal(r["state"][~mv], board[~mv]), a
        assert bool((res["reward"][:, a][~mv] == 0).all()) and bool((res["merged"][:, a][~mv] == 0).all())
        assert torch.equal(res["state"][:, a][~mv], board[~mv])
        env.load_state_dict(sd)


def _same_state(sd0: dict, sd1: dict) -> None:
    for k, t in sd0["tensors"].items():
        assert torch.equal(t, sd1["tensors"][k]), k
    for k, v in sd0["host"].items():
        if k == "schedule":
            assert type(v) is type(sd1["host"][k])
            continue
        if isinstance(v, np.ndarray):
            np.testing.assert_array_equal(v, sd1["host"][k])
        else:
            assert v == sd1["host"][k], k


@pytest.mark.gpu
@pytest.mark.parametrize("output", ["torch", "numpy"])
def test_vecgame_afterstates_equals_the_op_and_changes_nothing(ops, output):
    env = _played_env("improved", "replay", m=4097, steps=20)
    env.configure(output=output)
    want = _host(ops.afterstates(env._board[env._cur], reward_fn="improved", merged=True))
    sd0 = env.state_dict()
    epoch = env._state_epoch
    got = env.afterstates(merged=True)
    got2 = env.afterstates()
    assert set(got) == set(KEYS) and set(got2) == set(KEYS[:3])
    for k in KEYS:
        if output == "torch":
            assert got[k].is_cuda
            got[k] = got[k].cpu().numpy()
        assert isinstance(got[k], np.ndarray)
        np.testing.assert_array_equal(got[k], want[k], err_msg=k)
    _same_state(sd0, env.state_dict())
    assert env._state_epoch == epoch
    # the host generator is where it was: the next prepare() + step() equal those of an environment that never asked
    twin = _played_env("improved", "replay", m=4097, steps=20)
    twin.configure(output=output)
    for e in (env, twin):
        e.prepare()
    acts = np.random.default_rng(3).integers(0, 4, size=4097)
    ra, rb = env.step(acts.copy()), twin.step(acts.copy())
    for k in ("state", "reward", "valid_actions"):
        x, y = ra[k], rb[k]
        x = x.cpu().numpy() if isinstance(x, torch.Tensor) else x
        y = y.cpu().numpy() if isinstance(y, torch.Tensor) else y
        np.testing.assert_array_equal(x, y, err_msg=k)


# ---------------------------------------------------------------------------------------------
# sizes and memory safety
# ---------------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("m", [1, 3, 255, 256, 257, (1 << 20) + 3])
@pytest.mark.parametrize("dtype", [torch.uint8, torch.int8])
def test_sizes_against_the_oracle(ops, oracle, m, dtype):
    dev = _gpu()
    boards = _random_boards(m, seed=m)
    kind = KINDS[m % 4]
    for merged in (True, False):
        out, raw = _guarded_out(m, merged, dev)
        res = ops.afterstates(torch.from_numpy(boards).to(dev).view(dtype), reward_fn=kind, merged=merged, out=out)
        torch.cuda.synchronize()
        assert all(res[k] is out[k] for k in out)
        _canaries_intact(raw)
        host = _host(res)
        rows = np.arange(m) if m < 1024 else np.unique(np.r_[np.random.default_rng(m).integers(0, m, 4096), np.arange(m - 300, m)])
        _check_rows(oracle, boards, host, rows, kind)


def _tile_sum(x: torch.Tensor) -> torch.Tensor:
    x = x.long()
    return torch.where(x > 0, torch.ones_like(x) << x, torch.zeros_like(x)).sum(dim=-1)


@pytest.mark.gpu
def test_bench_size_properties_and_sample(ops, oracle):
    """M = 2^24: tile sums conserved, normal reward = sum merged[k] * 2^(k+1), mask = ops.valid_actions, and a seeded sample
    of 65 536 rows against the oracle."""
    m = 1 << 24
    dev = _gpu()
    boards_np = _random_boards(m, seed=24)
    board = torch.from_numpy(boards_np).to(dev)
    out, raw = _guarded_out(m, True, dev)
    res = ops.afterstates(board, merged=True, out=out)
    torch.cuda.synchronize()
    _canaries_intact(raw)
    want_sum = _tile_sum(board)
    for a in range(4):
        assert torch.equal(_tile_sum(res["state"][:, a]), want_sum), a
    w = torch.tensor([float(2 ** (k + 1)) for k in range(16)], dtype=torch.float64, device=dev)  # exact powers of two
    assert torch.equal((res["merged"].double() * w).sum(dim=-1), res["reward"].double())
    assert torch.equal(res["valid_actions"], ops.valid_actions(board))
    rows = np.random.default_rng(2024).choice(m, size=65536, replace=False)
    _check_rows(oracle, boards_np, _host(res), rows, "normal")


@pytest.mark.gpu
def test_beyond_32_bit_byte_offsets(ops, oracle):
    """M = 2^25 + 1: the afterstate of the last game sits 2^31 bytes into its buffer.  The guard before that buffer is 2 GiB
    long, so an offset that wrapped at 2^31 would land in it and be seen, not in someone else's memory."""
    m = (1 << 25) + 1
    dev = _gpu()
    boards_np = _random_boards(m, seed=25)
    out, raw = _guarded_out(m, False, dev, lead={"state": (1 << 31) + 256})
    res = ops.afterstates(torch.from_numpy(boards_np).to(dev), reward_fn="maxcell", out=out)
    torch.cuda.synchronize()
    _canaries_intact(raw)
    host = _host(res)
    rows = np.unique(np.r_[np.random.default_rng(25).integers(0, m, 2048), np.arange((1 << 25) - 64, m), np.arange(64)])
    _check_rows(oracle, boards_np, host, rows, "maxcell")


# ---------------------------------------------------------------------------------------------
# CUDA graph
# ---------------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("merged", [True, False])
def test_graph_replay_equals_eager(ops, merged):
    dev = _gpu()
    m = 50001
    static_board = torch.from_numpy(_random_boards(m, seed=1)).to(dev)
    static_out = {k: torch.empty((m,) + SHAPES[k][0], dtype=SHAPES[k][1], device=dev) for k in (KEYS if merged else KEYS[:3])}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.afterstates(static_board, reward_fn="improved", merged=merged, out=static_out)  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ops.afterstates(static_board, reward_fn="improved", merged=merged, out=static_out)
    for seed in (2, 3):
        static_board.copy_(torch.from_numpy(_random_boards(m, seed=seed)).to(dev))
        for t in static_out.values():
            t.view(torch.uint8).fill_(0x5A)
        graph.replay()
        want = ops.afterstates(static_board.clone(), reward_fn="improved", merged=merged)
        torch.cuda.synchronize()
        for k, t in static_out.items():
            assert torch.equal(t.view(torch.uint8), want[k].view(torch.uint8)), (seed, k)


# ---------------------------------------------------------------------------------------------
# argument checks
# ---------------------------------------------------------------------------------------------


def test_c_entry_argument_errors(lib):
    """Every error is returned before anything is launched, so this runs without a GPU."""
    p = 1 << 20  # 16-byte aligned stand-in device pointers: never dereferenced
    f = lib.ml2048_afterstates
    ok = dict(board=p, after=p + 4096, reward=p + 8192, valid=p + 12288, merged=p + 16384, kind=0, n=10)

    def call(**kw):
        a = {**ok, **kw}
        return f(a["board"], a["after"], a["reward"], a["valid"], a["merged"], a["kind"], a["n"], None)

    assert call(n=0) == -3 and call(n=-1) == -3
    assert call(n=0, board=None) == -3  # the size is checked first
    assert call(n=1 << 62) == -3        # more blocks than a grid holds
    for k in ("board", "after", "reward", "valid"):
        assert call(**{k: None}) == -1, k
    for k, off in (("board", 8), ("after", 4), ("merged", 8), ("reward", 2)):
        assert call(**{k: ok[k] + off}) == -2, k
    assert call(valid=ok["valid"] + 1, kind=-1) == -4  # bytes: any address passes the alignment checks
    for kind in (-1, 4, 1 << 20):
        assert call(kind=kind) == -4, kind
    assert call(kind=-1, reward=ok["reward"] + 2) == -2  # alignment before the enum


def test_python_argument_errors_without_a_gpu(ops):
    good = torch.zeros((8, 16), dtype=torch.uint8)
    with pytest.raises(ValueError, match="uint8/int8"):
        ops.afterstates(torch.zeros((8, 16), dtype=torch.int32))
    with pytest.raises(ValueError, match="uint8/int8"):
        ops.afterstates(torch.zeros((8, 15), dtype=torch.uint8))
    with pytest.raises(ValueError, match="uint8/int8"):
        ops.afterstates(torch.zeros((8, 4, 4), dtype=torch.uint8))
    with pytest.raises(ValueError, match="uint8/int8"):
        ops.afterstates(np.zeros((8, 16), np.uint8))
    with pytest.raises(ValueError, match="reward_fn"):
        ops.afterstates(good, reward_fn="shaped")
    with pytest.raises(ValueError, match="reward_fn"):
        ops.afterstates(good, reward_fn=lambda *a: 0.0)
    with pytest.raises(ValueError, match="dict"):
        ops.afterstates(good, out=[good])
    with pytest.raises(ValueError, match="does not write"):
        ops.afterstates(good, out={"next_state": good})
    with pytest.raises(ValueError, match="does not write"):
        ops.afterstates(good, out={"merged": torch.zeros((8, 4, 16), dtype=torch.uint8)})  # merged=False
    with pytest.raises(ValueError, match="CUDA"):
        ops.afterstates(good)
    with pytest.raises(ValueError, match="CUDA"):
        ops.afterstates(torch.zeros((16, 8), dtype=torch.uint8).t())


@pytest.mark.gpu
def test_python_argument_errors_on_the_device(ops):
    dev = _gpu()
    m = 8
    board = torch.zeros((m, 16), dtype=torch.uint8, device=dev)
    with pytest.raises(ValueError, match="CUDA"):
        ops.afterstates(torch.zeros((16, m), dtype=torch.uint8, device=dev).t())

    def good():
        return {k: torch.zeros((m,) + SHAPES[k][0], dtype=SHAPES[k][1], device=dev) for k in KEYS}

    bad = {
        "state": [torch.zeros((m, 64), dtype=torch.uint8, device=dev), torch.zeros((m, 4, 16), dtype=torch.int8, device=dev),
                  torch.zeros((m, 4, 16), dtype=torch.uint8), torch.zeros((m, 16, 4), dtype=torch.uint8, device=dev).transpose(1, 2),
                  torch.zeros((m + 1, 4, 16), dtype=torch.uint8, device=dev)],
        "reward": [torch.zeros((m, 4), dtype=torch.float64, device=dev), torch.zeros((m * 4,), dtype=torch.float32, device=dev),
                   torch.zeros((4, m), dtype=torch.float32, device=dev).t(), torch.zeros((m, 4), dtype=torch.float32)],
        "valid_actions": [torch.zeros((m, 4), dtype=torch.bool, device=dev), torch.zeros((m, 4), dtype=torch.uint8)],
        "merged": [torch.zeros((m, 4, 16), dtype=torch.int32, device=dev), torch.zeros((m, 4), dtype=torch.uint8, device=dev)],
        }
    for k, cases in bad.items():
        for t in cases:
            out = good()
            out[k] = t
            with pytest.raises(ValueError, match=k):
                ops.afterstates(board, merged=True, out=out)
    if torch.cuda.device_count() > 1:
        out = good()
        out["reward"] = out["reward"].to("cuda:1")
        with pytest.raises(ValueError, match="reward"):
            ops.afterstates(board, merged=True, out=out)
    res = ops.afterstates(board, merged=True, out=good())  # all good: empty boards, nothing moves
    assert int(res["valid_actions"].sum()) == 0 and int(res["state"].sum()) == 0
    assert ops.afterstates(torch.zeros((0, 16), dtype=torch.uint8, device=dev))["state"].shape == (0, 4, 16)
