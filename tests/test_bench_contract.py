"""bench.py's CPU-runnable arm must print exactly one JSON line with the contract's keys (the GPU arm is exercised on the
B200 box; its keys are checked here only statically)."""

from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tree_files() -> set:
    return {os.path.relpath(os.path.join(d, f), ROOT) for d, dirs, files in os.walk(ROOT) if ".git" not in d.split(os.sep)
            for f in files}


def test_reference_arm_prints_one_json_line():
    env = {k: v for k, v in os.environ.items() if k != "PYTHONDONTWRITEBYTECODE"}
    before = _tree_files()
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3",
                          "--cpu-games", "8192", "--ref-kind", "port"], check=True, capture_output=True, text=True, cwd=ROOT,
                         env=env).stdout
    assert _tree_files() == before  # bench.py writes nothing into the tree, not even bytecode of the modules it imports
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 3 and d["warmup"] >= 3
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None
    # --cpu-games sizes the CPU sample only: the config describes the GPU workload of the same command line
    assert d["config"]["games_per_gpu"] == d["config"]["global_games"] == 1 << 24


def test_reference_arm_times_the_staged_numba_reference():
    """`--impl reference` = the reference's own Numba VecGame (oracle/_ref) when it is staged and numba imports; its `config`
    is the GPU arm's config for the same command line (the driver compares them), the sample is described in cpu_baseline."""
    import pytest

    sys.path.insert(0, ROOT)
    import bench
    from oracle import make_ref

    if not make_ref.available():
        pytest.skip("oracle/_ref is not staged")
    pytest.importorskip("numba")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3",
                          "--cpu-games", "32768"], check=True, capture_output=True, text=True, cwd=ROOT).stdout
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["games"] == 32768 and cb["cores"] >= 1 and cb["value"] == d["value"] > 0
    assert "game_numba.py unmodified" in cb["sample"] and cb["step_only_value"] >= cb["value"]
    assert d["cpu_port"]["kind"] == "port" and d["cpu_port"]["value"] > 0
    ns = type("A", (), {"games_per_gpu": 1 << 24, "burn_in": bench.BURN_IN})()
    assert d["config"] == bench.make_config(ns, 1)  # what the GPU arm prints for the default command line
    assert d["steps"] == 3 and d["e2e"]["value"] == d["value"]


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr and r.stdout == ""


@pytest.mark.gpu
def test_dump_outputs_repeat_and_hold_the_last_step(tmp_path):
    """--dump-outputs: the same command line writes the same arrays (float32/float64, well under 64 MB), and they are the
    last timed step's: the dump of K steps differs from the dump of K + 1 steps."""
    m = 5000

    def run(steps: int, out: str) -> dict:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3",
                            "--games-per-gpu", str(m), "--burn-in", "40", "--no-extras", "--no-e2e", "--no-cpu-baseline",
                            "--no-shard-check", "--dump-outputs", str(tmp_path / out)],
                           check=True, capture_output=True, text=True, cwd=ROOT)
        assert json.loads(r.stdout)["steps"] == steps
        files = sorted(os.listdir(tmp_path / out))
        assert sum(os.path.getsize(tmp_path / out / f) for f in files) <= 64 << 20
        return {f[:-4]: np.load(tmp_path / out / f) for f in files}

    a, b, c = run(7, "a"), run(7, "b"), run(8, "c")
    assert {"state", "valid_actions", "reward", "terminated", "onehot", "id", "slot", "episode_stats"} <= set(a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert a["state"].shape == (m, 16) and a["onehot"].shape == (m, 16, 16)
    np.testing.assert_array_equal(a["slot"], np.arange(m))
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)
    np.testing.assert_array_equal(c["prev_state"][c["reset"] == 0], a["state"][c["reset"] == 0])
    assert not np.array_equal(a["state"], c["state"])


def _bench_gpu_arm(m: int, steps: int, out_dir) -> dict:
    args = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3", "--games-per-gpu", str(m),
            "--burn-in", "40", "--no-extras", "--no-e2e", "--no-cpu-baseline", "--no-shard-check"]
    if out_dir is not None:
        args += ["--dump-outputs", str(out_dir)]
    return json.loads(subprocess.run(args, check=True, capture_output=True, text=True, cwd=ROOT).stdout)


@pytest.mark.gpu
def test_dump_outputs_sample_a_larger_batch(tmp_path):
    """Above DUMP_GAMES games the dump is a seeded sample: sorted, distinct slots, the same ones on every run, and each
    sampled row is that slot's row of the whole batch after the last timed step (the batch replayed here in-process the
    way bench.py plays it)."""
    import torch

    import ml2048_b200

    sys.path.insert(0, ROOT)
    import bench

    m, steps = bench.DUMP_GAMES + 1000, 5
    _bench_gpu_arm(m, steps, tmp_path / "a")
    _bench_gpu_arm(m, steps, tmp_path / "b")
    a = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    b = {f[:-4]: np.load(tmp_path / "b" / f) for f in os.listdir(tmp_path / "b")}
    slot = a["slot"].astype(np.int64)
    assert slot.shape == (bench.DUMP_GAMES,) and np.all(np.diff(slot) > 0) and 0 <= slot[0] and slot[-1] < m
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)

    env = ml2048_b200.VecGame(m, ml2048_b200.reward_fn_normal, output="torch", onehot="f32", track_merged=False, sync_free=True)
    env.reset(0)
    for _ in range(40):
        env.prepare()
        env.step_random()
    for _ in range(3 + steps):
        env.step_random(auto_reset=True)
    board, valid = env.observations()
    sel = torch.from_numpy(slot).cuda()
    np.testing.assert_array_equal(a["state"], board[sel].cpu().numpy())
    np.testing.assert_array_equal(a["valid_actions"], valid[sel].cpu().numpy())
    np.testing.assert_array_equal(a["onehot"], env.observations_onehot()[sel].cpu().numpy())
    np.testing.assert_array_equal(a["id"], env._id[sel].cpu().numpy())
    np.testing.assert_array_equal(a["episode_stats"], env.episode_stats_tensor().cpu().numpy())


@pytest.mark.gpu
def test_both_arms_print_the_same_config():
    """The GPU arm and the CPU arm describe the same workload for the same command line."""
    gpu = _bench_gpu_arm(6000, 3, None)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--ref-kind", "port",
                          "--steps", "3", "--warmup", "3", "--games-per-gpu", "6000", "--burn-in", "40", "--cpu-games", "4096"],
                         check=True, capture_output=True, text=True, cwd=ROOT).stdout
    assert json.loads(out)["config"] == gpu["config"]
    assert gpu["config"]["games_per_gpu"] == 6000 and "burn-in" in gpu["config"]["workload"]


def test_other_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "3"],
                       check=True, capture_output=True, text=True, cwd=ROOT, env=env)
    assert r.stdout.strip() == ""


def test_gpu_arm_emits_the_contract_keys():
    src = open(os.path.join(ROOT, "bench.py")).read()
    for key in ('"metric"', '"value"', '"unit"', '"n_gpus"', '"steps"', '"warmup"', '"ms_per_step"', '"higher_is_better"',
                '"scaling"', '"vs_baseline"', '"dtype"', '"data"', '"config"', '"clocks"', '"e2e"', '"gpu_launches"', '"roofline"',
                '"cpu_baseline"', '"h2d_bytes_per_step"', '"d2h_bytes_per_step"', '"bound"', '"achieved"', '"peak"', '"frac"',
                '"traffic"', '"workload"', '"traffic_source"', '"shard_check"', '"collective_ms"', '"reduces_timed"',
                '"pcie_gbs"', '"pcie_ceiling_gbs"', '"cpu_port"'):
        assert key in src, key
