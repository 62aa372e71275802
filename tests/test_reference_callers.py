"""
The reference's OWN callers, unmodified, running on top of ``ml2048_b200.VecGame`` (the drop-in claim of INTEGRATION.md).

``oracle/_ref/ml2048`` is a byte-for-byte copy of the reference modules staged by ``oracle/make_ref.py`` (git-ignored test
infrastructure).  From it these tests import ``VecRunner`` + ``RunnerStats`` (runner.py:28-189), ``ReplayRecorder``
(replay.py:110-232), ``Policy`` / ``RandomPolicy`` (policy/) and hand them the CUDA environment in place of
``ml2048.game_numba.VecGame``:

  * the golden fixture ``runner_stack.npz`` was produced by exactly this stack around the reference VecGame
    (oracle/gen_golden.py:gen_runner) -- same policy, same seed -> the same histogram, per-id records and trajectories;
  * ``Trainer.on_stepped`` of run_train3.py:125-155 (the ``torch.from_numpy(result[k]).to(dtype)`` copies into the
    ``(use, step, game)`` buffers) and the ``eval_perf.py:66-102`` loop are replayed line for line;
  * ``_data[slot]["id"].item()`` (replay.py:147-151) is served from one host snapshot per prepare(), not nine gathers a slot.

CPU part (no GPU): the staged tree is intact and imports.  The ``_data`` lookup test needs no staged tree.
"""

from __future__ import annotations

import numpy as np
import pytest
import torch

from conftest import golden
from oracle import make_ref

needs_ref = pytest.mark.skipif(not make_ref.available(), reason="oracle/_ref is not staged (run python -m oracle.make_ref)")


@pytest.fixture(scope="module")
def refpkg():
    make_ref.import_reference()
    import ml2048.replay as replay
    import ml2048.runner as runner
    from ml2048 import game_numba
    from ml2048.policy import Policy
    from ml2048.policy.random import RandomPolicy

    return {"game_numba": game_numba, "runner": runner, "replay": replay, "Policy": Policy, "RandomPolicy": RandomPolicy}


def make_cycling_policy(Policy):
    class CyclingPolicy(Policy):
        """oracle/gen_golden.py:gen_runner -- k-th valid action with k = (7 t + 13 slot) mod nvalid; 0 when nothing is valid."""

        def __init__(self):
            super().__init__()
            self.t = 0

        def sample_actions(self, state, valid_actions, *, generator=None):
            m = valid_actions.shape[0]
            nvalid = valid_actions.sum(dim=1)
            k = (7 * self.t + 13 * torch.arange(m)) % nvalid.clamp(min=1)
            rank = torch.cumsum(valid_actions.long(), dim=1) - 1
            hit = valid_actions & (rank == k[:, None])
            actions = torch.where(nvalid > 0, hit.long().argmax(dim=1), torch.zeros(m, dtype=torch.long))
            self.t += 1
            return actions, torch.zeros(m)

    return CyclingPolicy()


@needs_ref
def test_staged_reference_is_intact_and_imports(refpkg):
    assert make_ref.available()
    gn = refpkg["game_numba"]
    import json

    with open(make_ref.MANIFEST) as fh:
        assert make_ref._sha(gn.__file__) == json.load(fh)["files"]["game_numba.py"]  # the unmodified reference, byte for byte
    assert gn.VecGame._DATA_DTYPE.itemsize == 64 and gn.VecGame._RAND_SIZE == 1024


@needs_ref
def test_reference_stack_on_the_oracle_reproduces_the_fixture(refpkg, oracle):
    """CPU: the same unmodified callers over the C oracle (VecGame surface) give the fixture too -- the harness itself is sound."""
    _run_stack_and_compare(refpkg, lambda m: oracle.OracleVecGame(m, "improved"))


def _run_stack_and_compare(refpkg, make_env):
    g = golden("runner_stack.npz")
    m, steps, seed = [int(x) for x in g["meta"]]
    VecRunner, RunnerStats = refpkg["runner"].VecRunner, refpkg["runner"].RunnerStats
    ReplayRecorder = refpkg["replay"].ReplayRecorder
    env = make_env(m)
    env.reset(seed)
    runner = VecRunner(env, 16, sample_device="cpu")
    stats = RunnerStats()
    rec = ReplayRecorder(10**9, 10**9, segment_size=64)
    runner.add_callback(VecRunner.EVENT_PREPARED, rec.on_prepared)
    runner.add_callback(VecRunner.EVENT_STEPPED, rec.on_stepped)
    runner.add_callback(VecRunner.EVENT_STEPPED, stats.on_stepped)
    runner.step_many(make_cycling_policy(refpkg["Policy"]), steps)
    bufs = sorted(rec.ready_buffers, key=lambda b: b.id)
    np.testing.assert_array_equal(stats.counts.astype(np.int64), g["stats_counts"])
    assert int(stats.terminated_count) == int(g["stats_terminated"])
    assert [(a, int(b)) for a, b, _ in env.summary()] == [tuple(r) for r in g["summary_live"].tolist()]
    assert int(env._game_count) == int(g["game_count"])
    np.testing.assert_array_equal(np.array([b.id for b in bufs]), g["buf_id"])
    np.testing.assert_array_equal(np.array([b.steps for b in bufs]), g["buf_steps"])
    np.testing.assert_array_equal(np.array([b.maxcell for b in bufs]), g["buf_maxcell"])
    np.testing.assert_array_equal(np.array([b.score for b in bufs], np.float32), g["buf_score"])
    by_id = {b.id: b for b in bufs}
    for gid in g["traj_ids"].tolist():
        st, ac, sc = by_id[gid].contiguous_result()
        np.testing.assert_array_equal(st, g[f"traj_{gid}_state"])
        np.testing.assert_array_equal(ac, g[f"traj_{gid}_action"])
        np.testing.assert_array_equal(sc, g[f"traj_{gid}_score"])
    return env


@pytest.mark.gpu
@needs_ref
def test_unmodified_vecrunner_runnerstats_replayrecorder_over_the_cuda_vecgame(refpkg):
    import ml2048_b200

    gn = refpkg["game_numba"]
    # reward_fn passed BY IDENTITY as run_train3.py:91-97 does: the reference's own njit function object
    _run_stack_and_compare(refpkg, lambda m: ml2048_b200.VecGame(m, gn.reward_fn_improved))


@pytest.mark.gpu
@needs_ref
def test_trainer_on_stepped_copies_and_lockstep_with_the_numba_reference(refpkg):
    """run_train3.py:112-157: VecRunner + RunnerStats + the trainer's ``on_stepped`` (its ``copy`` helper quoted verbatim)
    filling (use, step, game) REPLAY_SPEC buffers -- once around the live Numba VecGame, once around the CUDA one, with the
    reference's own RandomPolicy seeded identically.  Every buffer and the terminated-game statistics must be identical."""
    import ml2048_b200

    gn, REPLAY_SPEC = refpkg["game_numba"], refpkg["replay"].REPLAY_SPEC
    VecRunner, RunnerStats = refpkg["runner"].VecRunner, refpkg["runner"].RunnerStats
    m, steps, use = 512, 48, 2

    def run(env):
        torch.manual_seed(1234)  # RandomPolicy samples from torch's GLOBAL generator (policy/random.py:24, stats.py:32-47)
        env.reset(2024)
        runner = VecRunner(env, steps, sample_device="cpu")
        stats = RunnerStats()
        runner.add_callback(VecRunner.EVENT_STEPPED, stats.on_stepped)
        buffers = {k: torch.zeros((use, steps, m) + shape, dtype=dt) for k, (shape, dt) in REPLAY_SPEC.items()}
        state = {"epoch": 0, "si": 0}

        def on_stepped(game, result, actions, action_log_probs):
            ui = state["epoch"] % use
            si = state["si"]
            state["si"] += 1

            def copy(name: str, src: np.ndarray, dtype=None):  # run_train3.py:138-141
                src_tensor = torch.from_numpy(src).to(dtype=dtype)
                dst = buffers[name]
                dst[ui, si, ...].copy_(src_tensor)

            copy("state", result["prev_state"], torch.int8)
            copy("valid_actions", result["prev_valid_actions"], torch.bool)
            copy("next_state", result["state"], torch.int8)
            copy("next_valid_actions", result["valid_actions"], torch.bool)
            copy("reward", result["reward"], torch.float32)
            copy("terminated", result["terminated"], torch.bool)
            copy("step", result["step"], torch.int32)
            buffers["action"][ui, si, ...].copy_(actions.detach())
            buffers["action_log_prob"][ui, si, ...].copy_(action_log_probs.detach())

        runner.add_callback(VecRunner.EVENT_STEPPED, on_stepped)
        policy = refpkg["RandomPolicy"](seed=5)
        for epoch in range(use):
            state["epoch"], state["si"] = epoch, 0
            runner.step_many(policy, steps)
        return buffers, stats, env.summary()

    want, wstats, wsum = run(gn.VecGame(m, gn.reward_fn_improved))
    got, gstats, gsum = run(ml2048_b200.VecGame(m, gn.reward_fn_improved))
    for k in want:
        assert torch.equal(got[k], want[k]), k
    np.testing.assert_array_equal(gstats.counts, wstats.counts)
    assert int(gstats.terminated_count) == int(wstats.terminated_count) > 0
    assert [(a, int(b)) for a, b, _ in gsum] == [(a, int(b)) for a, b, _ in wsum]


@pytest.mark.gpu
@pytest.mark.parametrize("m", [3000, 65536, (1 << 20) + 1])
def test_data_view_serves_recorder_lookups_without_per_slot_round_trips(m):
    """replay.py:147-151 reads ``game._data[slot]["id"].item()`` per reset slot in a Python loop -- 65 536 times at
    eval_perf.py's first prepare().  The view serves them from ONE host snapshot (or, above 2^20 games, one gather per
    call), and fancy/slice/negative keys agree with the plain field arrays."""
    import ml2048_b200

    env = ml2048_b200.VecGame(m)
    env.reset(3)
    (idx,) = env.prepare()
    assert idx.size == m
    data = env._data
    torch.cuda.synchronize()
    ids = np.array(data["id"], copy=True)
    boards = np.array(data["board"], copy=True)
    import time

    n_look = min(m, 20000) if m <= (1 << 20) else 1000
    t0 = time.perf_counter()
    got = [data[int(s)]["id"].item() for s in idx[:n_look]]
    dt = time.perf_counter() - t0
    assert got == ids[:n_look].tolist()
    if m <= (1 << 20):
        assert dt / n_look < 80e-6, f"{dt / n_look * 1e6:.1f} us per lookup: the snapshot path is not being used"
    rec = data[-1]
    assert rec["id"].item() == ids[-1] and rec["board"].tolist() == boards[-1].tolist()
    sel = np.array([5, 0, m - 1, 17])
    np.testing.assert_array_equal(data[sel]["id"], ids[sel])
    np.testing.assert_array_equal(data[10:20]["board"], boards[10:20])
    mask = np.zeros(m, bool)
    mask[[1, 7, m - 2]] = True
    np.testing.assert_array_equal(data[mask]["id"], ids[mask])
    with pytest.raises(IndexError):
        data[m]
    # the snapshot follows the state: after a step the same view object returns the new records
    env.step(np.zeros(m, np.int64))
    np.testing.assert_array_equal(data[sel]["board"], np.asarray(env._data["board"])[sel])
    np.testing.assert_array_equal(data[sel]["step"], np.asarray(env._data["step"])[sel])


@pytest.mark.gpu
@needs_ref
def test_eval_perf_loop_over_the_cuda_vecgame(refpkg):
    """eval_perf.py:66-102 line for line (VecGame(batch), ReplayRecorder(batch, batch), VecRunner with both callbacks, the
    ``while remaining > 0`` drain of ``ready_buffers``), with the reference's RandomPolicy in place of the absent CNN
    checkpoint -- once on the Numba VecGame, once on the CUDA one: identical per-max-tile statistics."""
    import dataclasses
    from collections import defaultdict

    import ml2048_b200

    gn = refpkg["game_numba"]
    VecRunner, ReplayRecorder = refpkg["runner"].VecRunner, refpkg["replay"].ReplayRecorder

    @dataclasses.dataclass
    class StatEntry:
        count: int = 0
        score_sum: float = 0
        step_sum: int = 0

    def run(game_cls, rounds=600, batch_size=256):
        torch.manual_seed(4321)
        policy = refpkg["RandomPolicy"](seed=9)
        game = game_cls(batch_size)
        game.reset(77)  # eval_perf.py does not seed; seeded here so that both runs see the same tables
        recorder = ReplayRecorder(batch_size, batch_size)
        runner = VecRunner(game, batch_size, sample_device=None)
        runner.add_callback(VecRunner.EVENT_PREPARED, recorder.on_prepared)
        runner.add_callback(VecRunner.EVENT_STEPPED, recorder.on_stepped)
        stats = defaultdict(StatEntry)
        remaining = rounds
        runner_step = 0
        while remaining > 0:
            runner.step_once(policy)
            runner_step += 1
            while recorder.ready_buffers and remaining > 0:
                buffer = recorder.ready_buffers.popleft()
                if buffer.id >= rounds:
                    recorder.recording_threshold = 0
                    continue
                remaining -= 1
                key = 2 ** buffer.maxcell
                e = stats[key]
                e.count += 1
                e.step_sum += buffer.steps
                e.score_sum += buffer.score
        return {k: (v.count, v.step_sum, v.score_sum) for k, v in stats.items()}, runner_step

    base = gn.VecGame(1)._game_count  # fresh instances start their ids at 0 on both sides
    assert base == 0
    want, wsteps = run(gn.VecGame)
    got, gsteps = run(ml2048_b200.VecGame)
    assert got == want and gsteps == wsteps
    assert sum(c for c, _, _ in got.values()) == 600
