"""GPU tests of the rollout-path ops next to the environment (SURVEY.md section 8f): the kernel-written transition
record vs the reference's host copies, the masked categorical sampler vs torch, GAE vs the reference's compute_gae,
and the device runner."""

from __future__ import annotations

import numpy as np
import pytest
import torch

from conftest import golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ml():
    import ml2048_b200

    assert torch.cuda.is_available()
    return ml2048_b200


def test_gae_matches_reference_bit_exact(ml):
    """compute_gae of the live reference (tests/golden/gae.npz) -- bit-exact: same fp32 ops in the same order."""
    from ml2048_b200.ops import gae_advantages

    g = golden("gae.npz")
    for tag in "abc":
        gamma, lam = [float(x) for x in g[f"{tag}_params"]]
        t = {k: torch.from_numpy(g[f"{tag}_{k}"]).cuda() for k in ("v0", "v1", "reward", "terminated")}
        adv = gae_advantages(t["v0"], t["v1"], t["reward"], t["terminated"], gamma=gamma, lambda_=lam)
        np.testing.assert_array_equal(adv.cpu().numpy().view(np.uint32), g[f"{tag}_adv"].view(np.uint32), err_msg=tag)


def test_gae_matches_torch_at_training_shape(ml):
    """run_train3.py shape (use 2, step 16, game 4096) against the reference recurrence written in torch fp32."""
    from ml2048_b200.ops import gae_advantages

    torch.manual_seed(1)
    u, s, n = 2, 16, 4096
    v0, v1 = torch.randn(u, s, n, device="cuda") * 30, torch.randn(u, s, n, device="cuda") * 30
    reward = (torch.randint(0, 128, (u, s, n), device="cuda") * 4).float()
    term = torch.rand(u, s, n, device="cuda") < 0.01
    gamma, lam = 0.997, 0.95
    mask = ~term
    delta = gamma * v1 * mask + reward - v0  # gae.py:50
    tmp = torch.zeros(u, n, device="cuda")
    want = torch.empty_like(v0)
    for idx in reversed(range(s)):  # gae.py:65-68
        tmp = tmp * (gamma * lam)
        tmp = delta[:, idx, :] + tmp * mask[:, idx, :]
        want[:, idx, :] = tmp
    got = gae_advantages(v0, v1, reward, term, gamma=gamma, lambda_=lam)
    assert torch.equal(got, want)


def test_masked_categorical_log_probs_and_distribution(ml):
    """_sample_action (policy/actor_critic.py:56-76): log-probabilities against torch's Categorical within 1e-6 absolute
    (enough at randn*3 logits; test_rollout_numerics.py scales the tolerance with the logits), invalid actions never chosen,
    frequencies match softmax."""
    from ml2048_b200.ops import sample_masked_categorical

    torch.manual_seed(0)
    m = 1 << 18
    logits = torch.randn(m, 4, device="cuda") * 3
    valid = torch.rand(m, 4, device="cuda") < 0.7
    valid[:64] = False  # finished games: nothing valid
    actions, logp = sample_masked_categorical(logits, valid, seed=7, counter=3)
    min_real = torch.finfo(torch.float32).min
    masked = torch.where(valid, logits, min_real)
    dist = torch.distributions.Categorical(logits=masked)
    want_lp = dist.log_prob(actions)
    assert torch.allclose(logp, want_lp, rtol=0, atol=1e-6), (logp - want_lp).abs().max()
    any_valid = valid.any(dim=1)
    assert valid[any_valid].gather(1, actions[any_valid][:, None]).all()
    # one shared logit row sampled many times: empirical frequencies vs softmax
    row = torch.tensor([0.3, -1.2, 2.0, 0.7], device="cuda")
    mask = torch.tensor([True, True, False, True], device="cuda")
    acts, _ = sample_masked_categorical(row.repeat(m, 1), mask.repeat(m, 1), seed=11, counter=0)
    freq = torch.bincount(acts, minlength=4).double() / m
    p = torch.softmax(torch.where(mask, row, min_real).double(), dim=0)
    assert freq[2] == 0
    assert (freq - p).abs().max() < 4e-3
    # deterministic in (seed, counter); different counters give different draws
    a2, _ = sample_masked_categorical(logits, valid, seed=7, counter=3)
    a3, _ = sample_masked_categorical(logits, valid, seed=7, counter=4)
    assert torch.equal(a2, actions) and not torch.equal(a3, actions)


def test_step_from_logits_equals_sample_then_step(ml):
    """Sampling inside the step kernel == the stand-alone sampler followed by step(actions)."""
    from ml2048_b200.ops import sample_masked_categorical

    m = 5000
    fused = ml.VecGame(m, output="torch", sync_free=True)
    split = ml.VecGame(m, output="torch", sync_free=True)
    fused.reset(3)
    split.reset(3)
    torch.manual_seed(5)
    lp_f = torch.empty(m, device="cuda")
    for t in range(60):
        fused.prepare()
        split.prepare()
        logits = torch.randn(m, 4, device="cuda")
        counter = split._philox_counter  # the counter the step kernel is about to use
        acts, lp = sample_masked_categorical(logits, split.observations()[1], seed=split._philox_seed, counter=counter, dtype=torch.uint8)
        fused.step_from_logits(logits, log_prob_out=lp_f)
        split.step(acts)
        assert torch.equal(fused.sampled_actions, acts), t
        assert torch.equal(lp_f, lp), t
    assert torch.equal(fused.observations()[0], split.observations()[0])
    assert torch.equal(fused._score, split._score)


def test_transition_record_matches_trainer_copies(ml, oracle):
    """The kernel-written REPLAY_SPEC rows == what Trainer.on_stepped copies from the reference's results
    (run_train3.py:138-149), including stale reward/step/terminated on invalid moves."""
    from ml2048_b200.runner import RolloutBuffers
    from oracle.rollout import pick_actions

    m, steps = 1500, 48
    ref = oracle.OracleVecGame(m, "improved")
    ref.reset(8)
    env = ml.VecGame(m, ml.reward_fn_improved, output="torch", sync_free=True)
    env.reset(8)
    buf = RolloutBuffers(1, steps, m, "cuda")
    rng = np.random.default_rng(3)
    want = {k: [] for k in ("state", "valid_actions", "action", "reward", "next_state", "next_valid_actions", "step", "terminated")}
    for t in range(steps):
        ref.prepare()
        env.prepare()
        acts = pick_actions(ref.observations()[1], rng, wild=0.1)
        res = ref.step(acts)
        want["state"].append(res["prev_state"].astype(np.int8))
        want["valid_actions"].append(res["prev_valid_actions"].astype(bool))
        want["action"].append(acts.astype(np.int8))
        want["reward"].append(res["reward"].copy())
        want["next_state"].append(res["state"].astype(np.int8))
        want["next_valid_actions"].append(res["valid_actions"].astype(bool))
        want["step"].append(res["step"].copy())
        want["terminated"].append(res["terminated"].astype(bool))
        env.step(torch.from_numpy(acts).cuda(), record=buf.row(0, t))
    for k, rows in want.items():
        got = buf[k][0].cpu().numpy()
        exp = np.stack(rows)
        if exp.dtype == np.float32:
            got, exp = got.view(np.uint32), exp.view(np.uint32)
        np.testing.assert_array_equal(got, exp, err_msg=k)
    # after a step WITHOUT record the pointers are cleared: the buffers must not change any more
    snap = buf["next_state"].clone()
    env.prepare()
    env.step_random()
    assert torch.equal(buf["next_state"], snap)


@pytest.mark.parametrize("fused", [False, True])
def test_device_runner_drives_a_reference_style_policy(ml, fused):
    """DeviceRunner keeps VecRunner's surface (runner.py:28-117): callbacks, step_once/step_many, a Policy with
    sample_actions(state long, valid bool) -> (actions, log_probs); transitions land in the buffers."""
    from ml2048_b200.runner import DeviceRunner, DeviceRunnerStats, RolloutBuffers, UniformValidPolicy

    m, steps = 4096, 16
    env = ml.VecGame(m, ml.reward_fn_improved, output="torch")
    env.reset(0)
    buf = RolloutBuffers(2, steps, m, "cuda")
    runner = DeviceRunner(env, steps, buffers=buf, fused_sampler=fused)
    seen = {"prepared": 0, "stepped": 0, "new": 0}

    def on_prepared(game, new_indices):
        seen["prepared"] += 1
        seen["new"] += int(new_indices.numel())

    def on_stepped(game, result, actions, log_probs):
        seen["stepped"] += 1
        assert result["state"].shape == (m, 16) and actions.shape == (m,) and log_probs.shape == (m,)

    runner.add_callback(DeviceRunner.EVENT_PREPARED, on_prepared)
    runner.add_callback(DeviceRunner.EVENT_STEPPED, on_stepped)
    policy = UniformValidPolicy(seed=1)
    for epoch in range(12):
        runner.set_slot(epoch % 2, 0)
        runner.step_many(policy, steps)
    assert seen["prepared"] == seen["stepped"] == 12 * steps and seen["new"] >= m
    # consistency of the recorded rows: next_state of step t is the state of step t+1 unless the game was reset
    st, nx, term = buf["state"][1], buf["next_state"][1], buf["terminated"][1]
    same = (nx[:-1] == st[1:]).all(dim=-1)
    assert bool((same | term[:-1]).all())
    acts = buf["action"][1].long()
    assert bool(buf["valid_actions"][1].gather(-1, acts[..., None]).squeeze(-1)[~term.roll(1, 0)].float().mean() > 0.99)
    lp = buf["action_log_prob"][1]
    nvalid = buf["valid_actions"][1].sum(dim=-1).clamp(min=1)
    assert torch.allclose(lp[nvalid > 0], -torch.log(nvalid.float())[nvalid > 0], atol=1e-6)
    stats = DeviceRunnerStats(env)
    assert stats.terminated_count > 0 and sum(c for _, c, _ in stats.summary()) == stats.terminated_count


def test_whole_rollout_with_policy_as_one_cuda_graph(ml):
    """env kernels + a torch policy + in-kernel sampling + transition recording captured as ONE graph:
    replaying it equals the eager DeviceRunner rollout with the same policy and seeds."""
    from ml2048_b200.ops import encode_onehot
    from ml2048_b200.runner import DeviceRunner, RolloutBuffers

    torch.manual_seed(0)
    m, steps = 4096, 16
    net = torch.nn.Sequential(torch.nn.Linear(256, 64), torch.nn.Tanh(), torch.nn.Linear(64, 4)).cuda()

    def logits_fn(env):
        return net(encode_onehot(env.observations()[0]).flatten(1))

    class Policy:
        def action_logits(self, state, valid):
            return net(encode_onehot(state.to(torch.uint8)).flatten(1))

    eager = ml.VecGame(m, ml.reward_fn_improved, output="torch", sync_free=True)
    eager.reset(3)
    buf_e = RolloutBuffers(1, steps, m, "cuda")
    runner = DeviceRunner(eager, steps, buffers=buf_e, fused_sampler=True)
    graphed = ml.VecGame(m, ml.reward_fn_improved, output="torch", sync_free=True)
    graphed.reset(3)
    buf_g = RolloutBuffers(1, steps, m, "cuda")
    roll = ml.GraphedRollout(graphed, steps, window=steps * 4, logits_fn=logits_fn, buffers=buf_g)
    for epoch in range(6):
        runner.set_slot(0, 0)
        runner.step_many(Policy(), steps)
        roll.replay()
        torch.cuda.synchronize()
        for k in ("state", "action", "reward", "next_state", "terminated", "step", "valid_actions", "next_valid_actions"):
            assert torch.equal(buf_g[k], buf_e[k]), (epoch, k)
        assert torch.allclose(buf_g["action_log_prob"], buf_e["action_log_prob"], atol=1e-6)
    assert torch.equal(graphed.observations()[0], eager.observations()[0])
    assert graphed._game_count == eager._game_count


def test_trajectory_log_matches_replay_recorder(ml, oracle):
    """Device episode capture == ReplayRecorder's bookkeeping (replay.py:161-201) replayed on the host from the oracle's
    results: one (prev_state, action, score) row per runner step (invalid moves included), a final (state, 0, score) row."""
    from oracle.rollout import pick_actions

    m, n, cap, max_rows = 400, 600, 700, 512
    ref = oracle.OracleVecGame(m, "improved")
    ref.reset(6)
    env = ml.VecGame(m, ml.reward_fn_improved, output="torch")
    env.reset(6)
    env.enable_trajectory_log(cap, max_rows)
    rng = np.random.default_rng(2)
    rows = {}        # game id -> list of (state, action, score)
    finished = set()
    for t in range(n):
        ref.prepare()
        env.prepare()
        ids = ref._data["id"].copy()
        acts = pick_actions(ref.observations()[1], rng, wild=0.08)
        was_over = ref._data["terminated"].astype(bool).copy()
        res = ref.step(acts)
        env.step(torch.from_numpy(acts).cuda())
        for slot in range(m):
            gid = int(ids[slot])
            if gid >= cap or was_over[slot] or gid in finished:
                continue
            rows.setdefault(gid, []).append((res["prev_state"][slot].copy(), int(acts[slot]), float(res["score"][slot])))
            if res["terminated"][slot] and not res["invalid"][slot]:
                rows[gid].append((res["state"][slot].copy(), 0, float(res["score"][slot])))
                finished.add(gid)
    assert len(finished) > 300
    checked = 0
    for gid, want in rows.items():
        state, action, score = env.trajectory(gid)
        k = min(len(want), max_rows)
        assert state.shape[0] == k, (gid, state.shape[0], len(want))
        np.testing.assert_array_equal(state.cpu().numpy(), np.stack([w[0] for w in want[:k]]).astype(np.int8))
        np.testing.assert_array_equal(action.cpu().numpy(), np.array([w[1] for w in want[:k]], np.int8))
        np.testing.assert_array_equal(score.cpu().numpy(), np.array([w[2] for w in want[:k]], np.float32))
        checked += 1
    assert checked >= cap - 5


class _CyclingPolicy:
    """The deterministic policy of oracle/gen_golden.py::gen_runner, on the device."""

    def __init__(self):
        self.t = 0

    def sample_actions(self, state, valid_actions, *, generator=None):
        m = valid_actions.shape[0]
        nvalid = valid_actions.sum(dim=1)
        k = (7 * self.t + 13 * torch.arange(m, device=valid_actions.device)) % nvalid.clamp(min=1)
        rank = torch.cumsum(valid_actions.long(), dim=1) - 1
        hit = valid_actions & (rank == k[:, None])
        actions = torch.where(nvalid > 0, hit.long().argmax(dim=1), torch.zeros(m, dtype=torch.long, device=valid_actions.device))
        self.t += 1
        return actions, torch.zeros(m, device=valid_actions.device)


def test_device_runner_reproduces_the_reference_runner_stack(ml):
    """tests/golden/runner_stack.npz was produced by the reference's OWN VecRunner + RunnerStats + ReplayRecorder
    (runner.py, replay.py) around the reference VecGame.  The device runner with the same policy must give the same
    terminated-game histogram, the same per-game-id records (steps, max tile, score) and the same trajectories."""
    from ml2048_b200.runner import DeviceRunner, DeviceRunnerStats

    g = golden("runner_stack.npz")
    m, steps, seed = [int(x) for x in g["meta"]]
    env = ml.VecGame(m, ml.reward_fn_improved, output="torch")
    env.reset(seed)
    cap = int(g["game_count"])
    env.enable_episode_log(cap)
    env.enable_trajectory_log(1001, 512)
    runner = DeviceRunner(env, 16)
    runner.step_many(_CyclingPolicy(), steps)
    stats = DeviceRunnerStats(env)
    np.testing.assert_array_equal(stats.counts, g["stats_counts"])          # RunnerStats.counts (runner.py:150-166)
    assert stats.terminated_count == int(g["stats_terminated"])
    assert env._game_count == cap
    assert [(a, int(b)) for a, b, _ in env.summary()] == [tuple(r) for r in g["summary_live"].tolist()]
    log = env.episode_log()
    ids = torch.from_numpy(g["buf_id"]).cuda()
    np.testing.assert_array_equal(log["steps"][ids].cpu().numpy(), g["buf_steps"])      # RecordBuffer.steps
    np.testing.assert_array_equal(log["max_tile"][ids].cpu().numpy(), g["buf_maxcell"])  # RecordBuffer.maxcell
    np.testing.assert_array_equal(log["score"][ids].cpu().numpy(), g["buf_score"])       # RecordBuffer.score
    unfinished = torch.ones(cap, dtype=torch.bool, device="cuda")
    unfinished[ids] = False
    assert int(log["max_tile"][unfinished].sum()) == 0  # games the recorder had not finished are unfinished here too
    for gid in g["traj_ids"].tolist():                  # RecordBuffer.contiguous_result (replay.py:86-107)
        st, ac, sc = env.trajectory(gid)
        np.testing.assert_array_equal(st.cpu().numpy(), g[f"traj_{gid}_state"])
        np.testing.assert_array_equal(ac.cpu().numpy(), g[f"traj_{gid}_action"])
        np.testing.assert_array_equal(sc.cpu().numpy(), g[f"traj_{gid}_score"])
