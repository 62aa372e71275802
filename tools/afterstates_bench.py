"""Timing of the afterstates kernel (ops.afterstates: the four moves of every board, no spawn) against its byte floor.

    python tools/afterstates_bench.py [--sizes 16,20,22,24] [--iters 200] [--repeats 3] [--check-rows 4096] [--out FILE.json]

Boards come from a steady-state rollout (the in-kernel random policy with the auto-reset fused in, 400 steps).  For each
size, reward kind (normal, improved) and with / without `merged`, `iters` back-to-back launches are captured in one CUDA
graph and timed with CUDA events, `repeats` times (after a warm-up replay); the time per launch is the graph's time over
`iters`.  The byte floor is 16 B read + 64 + 16 + 4 B written = 100 B per board (164 B with `merged`) at the measured HBM
copy bandwidth (MEASURED_PEAKS.json hbm_gbs).  For context, step() with given actions (the kernel that moves one direction
and spawns) is timed at the same sizes.  A seeded sample of every timed output is checked against the C oracle in the same
run.  The device name and its power limit are printed with the numbers.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import ml2048_b200
from ml2048_b200 import ops


def hbm_gbs() -> tuple[float, str]:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (no MEASURED_PEAKS.json)"


def power_limit() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip() or "unknown"
    except Exception:
        return "unknown"


def steady_boards(m: int, steps: int) -> tuple[ml2048_b200.VecGame, torch.Tensor]:
    env = ml2048_b200.VecGame(m, output="torch", sync_free=True, track_merged=False)
    env.reset(0)
    for _ in range(steps):
        env.step_random(auto_reset=True)
    torch.cuda.synchronize()
    return env, env.observations()[0].clone()


def time_graph(fn, iters: int, repeats: int) -> list[float]:
    """us per call of `fn` over `iters` calls captured back to back in one CUDA graph, `repeats` replays."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()  # warm-up
    torch.cuda.synchronize()
    out = []
    for _ in range(repeats):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        g.replay()
        t1.record()
        t1.synchronize()
        out.append(t0.elapsed_time(t1) * 1e3 / iters)
    del g
    return out


def time_given_step(env: ml2048_b200.VecGame, iters: int) -> list[float]:
    """us per step(actions) (prepare() outside the timed window), actions recorded from the random policy on a snapshot."""
    snap = env.state_dict()
    acts = torch.empty((iters, env._size), dtype=torch.uint8, device=env.device)
    for t in range(iters):
        env.prepare()
        env.step_random(return_actions=True)
        acts[t].copy_(env.sampled_actions)
    env.load_state_dict(snap)
    env.prepare()
    env.step(acts[0])  # warm-up
    env.load_state_dict(snap)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for t in range(iters):
        env.prepare()
        ev[t][0].record()
        env.step(acts[t])
        ev[t][1].record()
    torch.cuda.synchronize()
    times = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
    return [times[0], times[len(times) // 2], times[-1]]


def check_sample(oracle, board_np: np.ndarray, res: dict, kind: str, rows: int, seed: int) -> int:
    idx = np.random.default_rng(seed).choice(board_np.shape[0], size=min(rows, board_np.shape[0]), replace=False)
    got = {k: v[torch.from_numpy(idx).to(v.device)].cpu().numpy() for k, v in res.items()}
    for j, i in enumerate(idx):
        b = board_np[i]
        for a in range(4):
            nb, mg = oracle.board_move(b, a)
            moved = bool((nb != b).any())
            want_r = oracle.board_reward(kind, nb, b, mg) if moved else 0.0
            ok = (got["state"][j, a] == nb).all() and got["valid_actions"][j, a] == moved and float(got["reward"][j, a]) == want_r
            if "merged" in got:
                ok = ok and (got["merged"][j, a] == mg).all()
            if not ok:
                raise AssertionError(f"row {i} direction {a} ({kind}) differs from the oracle")
    return len(idx)


def main() -> None:
    p = argparse.ArgumentParser()
    p.add_argument("--sizes", default="16,20,22,24", help="log2 of the board counts")
    p.add_argument("--iters", type=int, default=200, help="launches per timed CUDA graph (>= 100)")
    p.add_argument("--repeats", type=int, default=3)
    p.add_argument("--rollout-steps", type=int, default=400)
    p.add_argument("--check-rows", type=int, default=4096)
    p.add_argument("--out", default=None)
    a = p.parse_args()
    if a.iters < 100:
        raise SystemExit("--iters must be >= 100")
    if not torch.cuda.is_available():
        raise SystemExit("afterstates_bench.py needs a GPU")
    from oracle import oracle as orc

    orc.load_lib()
    peak, peak_src = hbm_gbs()
    meta = {"device": torch.cuda.get_device_name(0), "power_limit,max_sm_clock": power_limit(), "hbm_gbs": peak,
            "hbm_source": peak_src, "iters": a.iters, "repeats": a.repeats}
    print(json.dumps(meta))
    print("M <= 2^20: the 16 MiB of input boards (and at 2^16 the outputs too) sit in the 126 MB L2 across launches; "
          "2^22 and 2^24 stream from HBM")
    rows = []
    for lg in [int(x) for x in a.sizes.split(",")]:
        m = 1 << lg
        env, board = steady_boards(m, a.rollout_steps)
        board_np = board.cpu().numpy()
        valid_share = float(ops.valid_actions(board).float().mean())
        for kind in ("normal", "improved"):
            for merged in (False, True):
                keys = ("state", "reward", "valid_actions", "merged") if merged else ("state", "reward", "valid_actions")
                shapes = {"state": ((4, 16), torch.uint8), "reward": ((4,), torch.float32), "valid_actions": ((4,), torch.uint8),
                          "merged": ((4, 16), torch.uint8)}
                out = {k: torch.empty((m,) + shapes[k][0], dtype=shapes[k][1], device=board.device) for k in keys}
                us = time_graph(lambda: ops.afterstates(board, reward_fn=kind, merged=merged, out=out), a.iters, a.repeats)
                checked = check_sample(orc, board_np, out, kind, a.check_rows, seed=lg)
                per_board = 164 if merged else 100
                floor_us = m * per_board / (peak * 1e9) * 1e6
                r = {"M": m, "log2M": lg, "reward": kind, "merged": merged, "us": [round(x, 2) for x in us],
                     "gboards_per_s": round(m / min(us) / 1e3, 2), "bytes_per_board": per_board, "floor_us": round(floor_us, 2),
                     "floor_share": round(floor_us / min(us), 3), "achieved_gbs": round(m * per_board / min(us) / 1e3, 1),
                     "oracle_rows_checked": checked, "valid_share": round(valid_share, 4)}
                rows.append(r)
                print(json.dumps(r))
                del out
        st = time_given_step(env, a.iters)
        r = {"M": m, "log2M": lg, "kernel": "step(given actions)", "us_min_median_max": [round(x, 2) for x in st],
             "g_env_steps_per_s": round(m / st[1] / 1e3, 2)}
        rows.append(r)
        print(json.dumps(r))
        del env, board
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as fh:
            json.dump({"meta": meta, "rows": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
