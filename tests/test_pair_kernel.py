"""
The two-games-per-thread lean step kernel (``step_pair_kernel``: large batches without one-hot, ``merged`` or rollout extras)
against the one-game-per-thread kernel (``ML2048_STEP=single``) and against the CPU oracle: same arithmetic, same draws, so
every array must be bit-identical -- given actions, the in-kernel random policy, the fused auto-reset, both spawn modes, the
device schedule, odd batch sizes (the last thread owns ONE game) and sizes that end inside a warp.
"""

from __future__ import annotations

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

PAIR_MIN = 1 << 17  # kPairMinGames
STATE = ("_board", "_valid", "_id", "_step_score", "_reward", "_terminated_padded", "_invalid", "_reset_count_dev", "_game_count_dev")


@pytest.fixture(scope="module")
def ml():
    import ml2048_b200

    assert torch.cuda.is_available()
    return ml2048_b200


def same_state(a, b, what):
    assert a._cur == b._cur
    for name in STATE:
        assert torch.equal(getattr(a, name), getattr(b, name)), f"{name} {what}"
    # (the 64 replicas of the statistics are indexed by block, and the two kernels have different grids: compare the totals)
    assert torch.equal(a.episode_stats_tensor(), b.episode_stats_tensor()), f"episode statistics {what}"
    n = int(a._reset_count_dev.item())
    assert torch.equal(a._reset_indices_dev[:n], b._reset_indices_dev[:n]), f"reset indices {what}"


@pytest.mark.parametrize("rng_mode", ["replay", "philox"])
@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("m", [PAIR_MIN, PAIR_MIN + 1, PAIR_MIN + 37, (1 << 19) + 5, (1 << 20) + 77])
def test_pair_kernel_equals_single_kernel_random_policy(ml, monkeypatch, rng_mode, fused, m):
    kw = dict(rng_mode=rng_mode, output="torch", track_merged=False, sync_free=True)
    monkeypatch.setenv("ML2048_STEP", "pair")
    pair = ml.VecGame(m, "improved", **kw)
    single = ml.VecGame(m, "improved", **kw)
    pair.reset(3)
    single.reset(3)
    for t in range(160):
        for env, mode in ((pair, "pair"), (single, "single")):
            monkeypatch.setenv("ML2048_STEP", mode)
            if not fused:
                env.prepare()
            env.step_random(return_actions=True, auto_reset=fused)
        if t < 3 or t % 20 == 0 or t == 159:
            same_state(pair, single, f"step {t}")
            assert torch.equal(pair.sampled_actions, single.sampled_actions), t
    assert pair._game_count == single._game_count > m


@pytest.mark.parametrize("reward,two_prob", [("normal", 0.8), ("improved", 0.8), ("rank", 0.3), ("maxcell", 1.0)])
def test_pair_kernel_given_actions_against_the_oracle(ml, oracle, monkeypatch, reward, two_prob):
    """Lock step with the oracle, wrong directions included; the environment runs in scheduled mode for half of the steps."""
    monkeypatch.setenv("ML2048_STEP", "pair")
    m, n = PAIR_MIN + 3, 140
    ref = oracle.OracleVecGame(m, reward, two_prob=two_prob)
    ref.reset(21)
    env = ml.VecGame(m, reward, two_prob=two_prob, output="torch", track_merged=False)
    env.reset(21)
    acts = np.empty(m, np.int64)
    for t in range(n):
        if t == n // 2:
            env.schedule_ahead(n - t)
        (i0,) = ref.prepare()
        (i1,) = env.prepare()
        ref.random_valid_actions(500 + t, acts)
        if t % 3 == 0:
            acts[::7] = (acts[::7] + 1) % 4
        want = ref.step(acts)
        res = env.step(torch.from_numpy(acts.astype(np.int32 if t % 2 else np.int64)).cuda())
        if t < 2 or t % 20 == 0 or t == n - 1:
            assert torch.equal(i1, torch.from_numpy(i0).cuda()), t
            for k in ("state", "valid_actions", "step", "terminated", "invalid", "prev_state", "prev_valid_actions"):
                assert torch.equal(res[k], torch.from_numpy(np.ascontiguousarray(want[k])).cuda()), f"{k} step {t}"
            for k in ("reward", "score"):
                assert torch.equal(res[k].contiguous().view(torch.int32), torch.from_numpy(want[k].view(np.int32).copy()).cuda()), f"{k} step {t}"
            assert torch.equal(env._id, torch.from_numpy(ref._data["id"].copy()).cuda())
    assert env._game_count == ref._game_count


def test_pair_kernel_fused_rollout_against_the_oracle(ml, oracle, monkeypatch):
    monkeypatch.setenv("ML2048_STEP", "pair")
    m, n = PAIR_MIN + 1, 200
    env = ml.VecGame(m, "improved", output="torch", track_merged=False, sync_free=True)
    env.reset(8)
    ref = oracle.OracleVecGame(m, "improved")
    ref.reset(8)
    for t in range(n):
        res = env.step_random(return_actions=True, auto_reset=True)
        (want_idx,) = ref.prepare()
        want = ref.step(env.sampled_actions.cpu().numpy().astype(np.int64))
        if t < 2 or t % 25 == 0 or t == n - 1:
            (got_idx,) = env.last_reset()
            np.testing.assert_array_equal(got_idx.cpu().numpy(), want_idx)
            for k in ("state", "valid_actions", "step", "terminated", "invalid", "prev_state", "prev_valid_actions"):
                np.testing.assert_array_equal(res[k].cpu().numpy(), want[k], err_msg=f"{k} step {t}")
            np.testing.assert_array_equal(res["score"].cpu().numpy().view(np.uint32), want["score"].view(np.uint32))
            np.testing.assert_array_equal(env._id.cpu().numpy(), ref._data["id"])
    assert env._game_count == ref._game_count > 2 * m


@pytest.mark.parametrize("rng_mode", ["replay", "philox"])
@pytest.mark.parametrize("fused", [False, True])
def test_pair_kernel_graph_replay_equals_eager(ml, monkeypatch, rng_mode, fused):
    """The in-kernel policy from the device schedule inside a CUDA graph: a step draws with the Philox counter after its
    prepare()'s, exactly as in eager mode."""
    monkeypatch.setenv("ML2048_STEP", "pair")
    m, steps, replays = PAIR_MIN + 3, 8, 8
    kw = dict(rng_mode=rng_mode, output="torch", track_merged=False, sync_free=True)
    eager = ml.VecGame(m, "improved", **kw)
    eager.reset(5)
    for _ in range(steps * replays):
        if not fused:
            eager.prepare()
        eager.step_random(auto_reset=fused)
    env = ml.VecGame(m, "improved", **kw)
    env.reset(5)
    roll = ml.GraphedRollout(env, steps, window=steps * 3, auto_reset=fused)
    roll.replay(replays)
    torch.cuda.synchronize()
    same_state(eager, env, "graph replay")
    assert env._game_count == eager._game_count > m


@pytest.mark.parametrize("rng_mode", ["replay", "philox"])
def test_pair_kernel_shard_at_an_odd_slot(ml, monkeypatch, rng_mode):
    """A Philox block serves a PAIR of global slots (slot >> 1).  A shard that starts at an odd global slot has its threads'
    two games in two different blocks: its draws (policy words, Philox spawn cells) must still be those of the whole batch."""
    monkeypatch.setenv("ML2048_STEP", "pair")
    cut = PAIR_MIN + 1  # odd: the second shard's first slot
    m = cut + PAIR_MIN + 2
    kw = dict(rng_mode=rng_mode, output="torch", track_merged=False, sync_free=True)
    whole = ml.VecGame(m, "improved", **kw)
    parts = [ml.VecGame(cut, "improved", slot_base=0, **kw), ml.VecGame(m - cut, "improved", slot_base=cut, **kw)]
    for e in [whole] + parts:
        e.reset(17)
    for t in range(130):
        for e in [whole] + parts:
            e.step_random(return_actions=True, auto_reset=True)
        if t < 2 or t % 32 == 0 or t == 129:
            for name in ("_step_score", "_reward", "_invalid"):
                assert torch.equal(torch.cat([getattr(p, name) for p in parts]), getattr(whole, name)), (name, t)
            assert torch.equal(torch.cat([p._terminated_padded[: p._size] for p in parts]), whole._terminated_padded[:m]), t
            assert torch.equal(torch.cat([p.sampled_actions for p in parts]), whole.sampled_actions), t
            for k in (0, 1):
                assert torch.equal(torch.cat([p.observations()[k] for p in parts]), whole.observations()[k]), (k, t)
    assert whole.episode_stats()["episodes"] == sum(p.episode_stats()["episodes"] for p in parts) > m // 4
