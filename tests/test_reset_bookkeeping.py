"""The integer bookkeeping of the auto-reset on the GPU against the plain NumPy definition (tests/_reset_ref.py): which
games reset, in which order, and with which ids -- at the sizes where the single-block scans carry a running total from
one pass of 1024 entries to the next.

    (a) ml2048_autoreset_scan through the C ABI: every output vs scan_ref, up to three passes over the chunk totals
        (> 2^26 games), with and without id_offset, canary words around every buffer
    (b) the fused auto-reset above one pass (2^25 + 33 games = 1025 chunks), pair and one-game kernels, vs prepare() + step
        and vs prepare_ref
    (c) prepare() beyond 1024 tiles and at the edge of the single-block kernel, split and default path, vs prepare_ref
    (d) the sharded prepare (count, all-gather, apply with id_offset) of three shards of > 1024 tiles each, emulated in one
        process, vs the whole batch
    (e) ml2048_max_tile_hist with a `terminated` array vs np.bincount
"""

from __future__ import annotations

import gc

import numpy as np
import pytest
import torch

import _reset_ref as ref
from test_fused_autoreset import assert_same_state
from test_guard_bands import Arena

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ml():
    import ml2048_b200

    assert torch.cuda.is_available()
    return ml2048_b200


def _dev(a: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(autouse=True)
def _release_memory():
    """Hands the memory of a test's environments (a few GB at these sizes) back to the device when it ends."""
    yield
    gc.collect()
    torch.cuda.empty_cache()


# ---- (a) the scan alone -------------------------------------------------------------------------------------------------

SCAN_SIZES = [1, 16, 17, 32, 33, 32767, 32768, 32769, 1 << 25, (1 << 25) + 1, (1 << 26) + (1 << 15) + 7]
GAME_COUNT0 = 123_456_789
ID_OFFSET = 987_654_321


@pytest.mark.parametrize("m", SCAN_SIZES)
def test_autoreset_scan_against_numpy(ml, m):
    """Every output of ml2048_autoreset_scan for every flag pattern, several calls in a row on one scratch buffer: the
    ranks, the chunk bases, the id base and count, the id counter (advanced from a non-zero start, or left alone when
    id_offset is set); the flags stay as they were, the ticket word returns to 0, nothing is written outside the outputs."""
    from ml2048_b200 import _lib

    lib = _lib.load()
    groups = -(-m // ref.GROUP)
    chunks = -(-groups // ref.CHUNK)
    if m == SCAN_SIZES[-1]:
        assert chunks > 2 * ref.CHUNK  # three passes over the chunk totals
    n_scratch = int(lib.ml2048_autoreset_scratch_ints(m))
    assert n_scratch >= chunks + 1
    pad = -(-m // 16) * 16
    ar = Arena(pad + 4 * (groups + chunks + n_scratch) + 4 * 8 + 20 * 4096 + 8 * 512)
    flags = ar.take(pad)
    rank = ar.take(4 * groups, torch.int32)
    chunk_base = ar.take(4 * chunks, torch.int32)
    scratch = ar.take(4 * n_scratch, torch.int32)  # zero before the first call
    game_count, id_offset = ar.take(8, torch.int64), ar.take(8, torch.int64)
    id_base, count = ar.take(8, torch.int64), ar.take(8, torch.int64)
    id_offset.fill_(ID_OFFSET)
    stream = torch.cuda.current_stream().cuda_stream
    for k, name in enumerate(ref.PATTERNS):
        f = ref.flag_pattern(name, m, seed=k)
        want = ref.scan_ref(f)
        flags[:m].copy_(_dev(f))
        before = flags.clone()
        for sharded in (False, True):
            what = f"{name}, id_offset={sharded}"
            for out in (rank, chunk_base, id_base, count):
                out.view(torch.uint8).fill_(0xEE)  # every entry must be written
            game_count.fill_(GAME_COUNT0 + k)
            rc = lib.ml2048_autoreset_scan(flags.data_ptr(), rank.data_ptr(), chunk_base.data_ptr(), m, game_count.data_ptr(),
                                           id_offset.data_ptr() if sharded else None, id_base.data_ptr(), count.data_ptr(),
                                           scratch.data_ptr(), stream)
            _lib.check(rc, "ml2048_autoreset_scan")
            np.testing.assert_array_equal(rank.cpu().numpy(), want.reset_rank, err_msg=f"reset_rank {what}")
            np.testing.assert_array_equal(chunk_base.cpu().numpy(), want.reset_chunk_base, err_msg=f"reset_chunk_base {what}")
            assert int(count.item()) == want.total, what
            assert int(id_base.item()) == GAME_COUNT0 + k + (ID_OFFSET if sharded else 0), what
            assert int(game_count.item()) == GAME_COUNT0 + k + (0 if sharded else want.total), what
            assert int(id_offset.item()) == ID_OFFSET, what
            assert int(scratch[chunks].item()) == 0, f"ticket {what}"
            assert torch.equal(flags, before), f"flags {what}"
    ar.check()


# ---- (b) the fused auto-reset above one pass of the scan ----------------------------------------------------------------

FUSED_M = (1 << 25) + 33  # 1025 chunks; ends inside a warp; odd, so the last thread of the pair kernel owns one game
FUSED_PATTERNS = ("chunk1024", "last", "first_of_chunk", "random1")


def test_dead_board_is_dead(ml):
    from ml2048_b200 import _lib

    lib = _lib.load()
    board = _dev(np.tile(ref.DEAD_BOARD, (3, 1)))
    valid = torch.full((3, 4), 7, dtype=torch.uint8, device="cuda")
    _lib.check(lib.ml2048_valid_actions(board.data_ptr(), valid.data_ptr(), 3, torch.cuda.current_stream().cuda_stream),
               "ml2048_valid_actions")
    assert int(valid.sum()) == 0


@pytest.mark.parametrize("kernel,rng_mode", [("pair", "replay"), ("single", "replay"), ("pair", "philox")])
def test_fused_autoreset_beyond_one_scan_pass(ml, monkeypatch, kernel, rng_mode):
    """step_random(auto_reset=True) against prepare() + step_random() at 1025 chunks: the first step after reset() resets
    every game, then the same slots of both environments are ended on purpose (dead board, zero mask, terminated) before
    one step.  The two stay equal, and the reset slots, their ids and the id counter are prepare_ref's."""
    monkeypatch.setenv("ML2048_STEP", kernel)
    m = FUSED_M
    assert -(-(-(-m // ref.GROUP)) // ref.CHUNK) == ref.CHUNK + 1
    kw = dict(rng_mode=rng_mode, output="torch", track_merged=False, sync_free=True)
    plain = ml.VecGame(m, "improved", **kw)
    fused = ml.VecGame(m, "improved", **kw)
    plain.reset(13)
    fused.reset(13)
    dead = _dev(ref.DEAD_BOARD)
    for k, name in enumerate((None,) + FUSED_PATTERNS):
        if name is not None:
            slots = _dev(np.flatnonzero(ref.flag_pattern(name, m, seed=k)))
            for env in (plain, fused):
                env._board[env._cur][slots] = dead
                env._valid[env._cur][slots] = 0
                env._terminated[slots] = 1
        flags = fused._terminated.cpu().numpy()
        want = ref.prepare_ref(flags, fused._game_count)
        if name is None:
            assert want.n == m
        plain.prepare()
        plain.step_random()
        fused.step_random(auto_reset=True)
        what = f"{kernel} {rng_mode} {name or 'after reset()'}"
        assert_same_state(plain, fused, what)
        n = int(fused._reset_count_dev.item())
        assert n == want.n, what
        idx = fused._reset_indices_dev[:n]
        assert torch.equal(idx, _dev(want.indices)), what
        assert torch.equal(fused._id[idx].long(), _dev(want.ids)), what
        assert fused._game_count == want.game_count, what


# ---- (c) prepare() beyond 1024 tiles -------------------------------------------------------------------------------------

PREPARE_PATTERNS = ("tile1024", "first_of_tile", "last", "random1", "all")


@pytest.mark.parametrize("m", [8192, 8193, (1 << 22) + 2, (1 << 24) + 3])
def test_prepare_bookkeeping_against_numpy(ml, monkeypatch, m):
    """After a few steps `terminated` is overwritten with a pattern and prepare() runs, once under ML2048_PREPARE=split
    (above 8192 games: count, scan, apply) and once on the default path (the single-block kernel up to 8192 games, else
    the cooperative one).  Index list, ids of the reset slots, id counter and reset count are prepare_ref's, the flags are
    cleared, the reset slots' records are zeroed and every other slot is bitwise untouched; both paths leave the same
    boards and masks."""
    envs = {}
    for path in ("split", "default"):
        env = ml.VecGame(m, "improved", output="torch", track_merged=False, sync_free=True)
        env.reset(21)
        envs[path] = env

    def on_path(path):
        if path == "split":
            monkeypatch.setenv("ML2048_PREPARE", "split")
        else:
            monkeypatch.delenv("ML2048_PREPARE", raising=False)

    fields = ("_id", "_step_score", "_reward", "_invalid", "_board", "_valid")

    def records(env):  # the reward compared bit for bit; board and mask of the current ping-pong half
        return {"_id": env._id, "_step_score": env._step_score, "_reward": env._reward.view(torch.int32),
                "_invalid": env._invalid, "_board": env._board[env._cur], "_valid": env._valid[env._cur]}

    for k, name in enumerate(("warm-up",) * 3 + PREPARE_PATTERNS):
        for path, env in envs.items():
            on_path(path)
            if name == "warm-up":
                env.prepare()
                continue
            what = f"{name} on the {path} path"
            # the pattern on top of the games that are over anyway
            f = ref.flag_pattern(name, m, seed=k) | env._terminated.cpu().numpy()
            env._terminated.copy_(_dev(f))
            want = ref.prepare_ref(f, env._game_count)
            mask = _dev(f).bool()
            keep = ~mask
            before = {field: t.clone() for field, t in records(env).items()}
            env.prepare()
            n = int(env._reset_count_dev.item())
            assert n == want.n, what
            assert env._game_count == want.game_count, what
            idx = env._reset_indices_dev[:n]
            assert torch.equal(idx, _dev(want.indices)), what
            assert torch.equal(env._id[idx].long(), _dev(want.ids)), what
            assert int(env._terminated_padded.count_nonzero()) == 0, what
            after = records(env)
            for field in fields:
                assert torch.equal(after[field][keep], before[field][keep]), f"{field} of the other slots, {what}"
            for field in ("_step_score", "_reward", "_invalid"):
                assert int(after[field][mask].count_nonzero()) == 0, f"{field} of the reset slots, {what}"
            del before, after
        if name != "warm-up":
            a, b = envs["split"], envs["default"]
            assert torch.equal(a._board[a._cur], b._board[b._cur]), f"boards after {name}"
            assert torch.equal(a._valid[a._cur], b._valid[b._cur]), f"masks after {name}"
        for env in envs.values():
            env.step_random()


# ---- (d) the sharded prepare, emulated in one process --------------------------------------------------------------------

SHARD_TOTAL = 3 * (1 << 22) + 4
SHARD_ROUNDS = 30


@pytest.mark.parametrize("rng_mode", ["replay", "philox"])
def test_sharded_prepare_equals_whole_batch(ml, monkeypatch, rng_mode):
    """Three shards of one batch of 3 * 2^22 + 4 games (> 1024 tiles each; the third starts at an odd slot), each
    prepare()d as a rank of a multi-GPU run does it -- ml2048_prepare_count, an all-gather of the per-shard counts (here the
    counts the test takes from the flags), ml2048_prepare_apply with id_offset -- against the same batch as ONE VecGame.
    30 rounds from reset(): 1 % extra resets every other round on top of the games that end by themselves, and one round
    each with resets in the last shard only and in the first shard only."""
    import torch.distributed as dist

    from ml2048_b200.sharding import shard_bounds

    world = 3
    bounds = [shard_bounds(SHARD_TOTAL, world, r) for r in range(world)]
    assert bounds == [(0, (1 << 22) + 2), ((1 << 22) + 2, (1 << 22) + 1), ((1 << 23) + 3, (1 << 22) + 1)]
    kw = dict(rng_mode=rng_mode, output="torch", track_merged=False, sync_free=True)
    whole = ml.VecGame(SHARD_TOTAL, **kw)
    shards = []
    for r, (base, size) in enumerate(bounds):
        s = ml.VecGame(size, slot_base=base, **kw)
        # what shard() sets, without a process group
        s._dist_group, s._dist_rank, s._dist_world = "emulated", r, world
        s._counts_all = torch.zeros((world,), dtype=torch.int64, device=s.device)
        shards.append(s)
    counts = []

    def all_gather_into_tensor(out, inp, group=None):
        assert group == "emulated" and out.shape == (world,) and inp.shape == (1,)
        out.copy_(torch.tensor(counts, dtype=torch.int64))

    monkeypatch.setattr(dist, "all_gather_into_tensor", all_gather_into_tensor)
    for env in [whole] + shards:
        env.reset(29)
    # the second shard is left without resets in the crafted rounds
    only_in = {1: 2, 2: 0}
    for t in range(SHARD_ROUNDS):
        if t in only_in:
            assert int(whole._terminated.count_nonzero()) == 0  # a move or two after reset(): no game can be over yet
            base, size = bounds[only_in[t]]
            f = np.zeros(SHARD_TOTAL, np.uint8)
            f[base:base + size] = ref.flag_pattern("first_of_tile", size) | ref.flag_pattern("tile1024", size)
        elif t % 2:
            f = ref.flag_pattern("random1", SHARD_TOTAL, seed=t)
        else:
            f = None
        if f is not None:
            fd = _dev(f).bool()
            whole._terminated[fd] = 1
            for s, (base, size) in zip(shards, bounds):
                s._terminated[fd[base:base + size]] = 1
        counts[:] = [int(s._terminated.sum()) for s in shards]
        assert sum(counts) == int(whole._terminated.sum())
        if t in only_in:
            assert [c > 0 for c in counts] == [r == only_in[t] for r in range(world)]
        whole.prepare()
        for s in shards:
            s.prepare()
        what = f"{rng_mode} round {t}"
        for s, c in zip(shards, counts):
            assert int(s._reset_count_dev.item()) == c, what
            assert s._game_count == whole._game_count, what
        n = int(whole._reset_count_dev.item())
        got = torch.cat([s._reset_indices_dev[:c] + base for s, c, (base, _) in zip(shards, counts, bounds)])
        assert torch.equal(got, whole._reset_indices_dev[:n]), what
        whole.step_random()
        for s in shards:
            s.step_random()
        for name in ("_id", "_step_score", "_terminated", "_invalid"):
            assert torch.equal(torch.cat([getattr(s, name) for s in shards]), getattr(whole, name)), f"{name} {what}"
        for name in ("_board", "_valid"):
            assert torch.equal(torch.cat([getattr(s, name)[s._cur] for s in shards]), getattr(whole, name)[whole._cur]), f"{name} {what}"
        stats = torch.stack([s.episode_stats_tensor() for s in shards])
        folded = torch.cat([stats[:, :23].sum(dim=0), stats[:, 23:].max(dim=0).values])
        assert torch.equal(folded, whole.episode_stats_tensor()), f"episode statistics {what}"


# ---- (e) the max-tile histogram of finished games ------------------------------------------------------------------------


def test_max_tile_hist_with_terminated(ml):
    """ml2048_max_tile_hist in its _update_count form (a `terminated` array; any non-zero byte counts) and without one,
    accumulated onto counts already in hist20, against np.bincount; more games than one pass of the grid-stride loop."""
    from ml2048_b200 import _lib

    lib = _lib.load()
    m = 3 * 148 * 8 * 256 + 5
    rng = np.random.default_rng(17)
    caps = np.where(rng.random(m) < 0.1, 255, rng.integers(0, 23, m))
    boards = (rng.random((m, 16)) * (caps[:, None] + 1)).astype(np.uint8)  # largest cell near the row's cap, up to 255
    term = rng.choice(np.array([0, 1, 2, 255], np.uint8), m, p=[0.4, 0.2, 0.2, 0.2])
    start = rng.integers(0, 1 << 40, 20).astype(np.uint64)
    bins = np.minimum(boards.max(axis=1), 19)
    assert (np.bincount(bins, minlength=20) > 0).all()
    want = start + np.bincount(bins[term != 0], minlength=20).astype(np.uint64)
    board_d, term_d = _dev(boards), _dev(term)
    hist = _dev(start.view(np.int64))
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.ml2048_max_tile_hist(board_d.data_ptr(), term_d.data_ptr(), m, hist.data_ptr(), stream), "ml2048_max_tile_hist")
    np.testing.assert_array_equal(hist.cpu().numpy().view(np.uint64), want)
    _lib.check(lib.ml2048_max_tile_hist(board_d.data_ptr(), None, m, hist.data_ptr(), stream), "ml2048_max_tile_hist")
    np.testing.assert_array_equal(hist.cpu().numpy().view(np.uint64), want + np.bincount(bins, minlength=20).astype(np.uint64))
    assert torch.equal(term_d, _dev(term)) and torch.equal(board_d, _dev(boards))
