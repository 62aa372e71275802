"""Multi-stage n-tuple networks (the ``stages=`` argument of ops.ntuple_*, NTupleNetwork(stages=...)): what a staged kernel
costs against the single-stage one, and how staged TD(0) / TD(lambda) learn against the single-stage network.

    python tools/stages_bench.py [--out-dir DIR] [--quick]

- Kernel cost: ntuple_value, ntuple_greedy, ntuple_td_update, ntuple_tc_update and ntuple_expectimax (depth 1) with
  S = 3 (stages (6, 7): the played boards below fall in all three stages; the share of each is reported) against S = 1, the
  standard 4x6 network with seeded random weights (S * 256 MiB), at M = 2^16, 2^18 and 2^20.  Boards: steady-state boards of
  the in-kernel random policy (400 steps with auto-reset at the largest size, smaller sizes take a prefix), as
  tools/lambda_bench.py builds them.  Each op is timed as a CUDA-graph replay of back-to-back calls (ntuple_bench's
  time_graph: CUDA events, one warm-up call outside the graph), S = 1 and S = 3 alternating, 5 rounds; the figure is the
  minimum over rounds and the ratio S = 3 / S = 1 of those minima.  A third network, S = 2 with stages (15,), puts every
  played board in stage 0: it runs the staged kernels' extra instructions over the single-stage network's table footprint,
  which separates the cost of the stage arithmetic from the cost of spreading the lookups over S tables.  Updates run with alpha = 1e-9 so that repeated calls
  leave the weights as they are up to rounding.
- Learning: M = 2^14, seed 0, 200 000 learner steps from zero weights, windows of 20 000 steps (ntuple_bench's
  learner_run): TD(0) with stages (), (10,) and (11,) at its default alpha, then TD(lambda) with h = 3, lambda = 0.25 at the
  split with the better final mean score; at equal steps and at equal wall time (the single-stage window that ends last at or
  before each staged window's time).
Device name and power limit are read in the same run.  Writes stages_bench.{json,txt} under --out-dir (default profiles/).
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch

from ntuple_bench import device_info, learner_run, time_graph

import ml2048_b200
from ml2048_b200 import ops
from ml2048_b200.ntuple import DEFAULT_ALPHA_TIMES_GAMES, STANDARD_4X6, NTupleNetwork

LINES: list = []
TIMED_STAGES = (6, 7)
ONE_TABLE_STAGES = (15,)  # S = 2, every played board in stage 0


def say(msg: str) -> None:
    LINES.append(msg)
    print(msg, flush=True)


def steady_boards(m: int) -> torch.Tensor:
    env = ml2048_b200.VecGame(m, output="torch", sync_free=True, track_merged=False)
    env.reset(0)
    for _ in range(400):
        env.step_random(auto_reset=True)
    torch.cuda.synchronize()
    b = env.observations()[0].clone()
    del env
    return b


def stage_shares(boards: torch.Tensor, stages) -> list:
    m = boards.to(torch.int32).clamp(max=15).amax(dim=1)
    st = sum((m >= t).to(torch.int64) for t in stages)
    return [float((st == s).float().mean()) for s in range(len(stages) + 1)]


def op_fns(b: torch.Tensor, stages, w: torch.Tensor, c: torch.Tensor, acc: torch.Tensor) -> dict:
    m = b.shape[0]
    dev = b.device
    target = torch.ones(m, device=dev)
    delta = torch.empty(m, device=dev)
    value = torch.empty(m, device=dev)
    g_out = {"action": torch.empty(m, dtype=torch.uint8, device=dev), "state": torch.empty((m, 16), dtype=torch.uint8, device=dev),
             "reward": torch.empty(m, device=dev), "value": torch.empty(m, device=dev)}
    x_out = dict(g_out, q=torch.empty((m, 4), device=dev))
    kw = {"stages": stages}
    return {
        "value": lambda: ops.ntuple_value(b, w, STANDARD_4X6, out=value, **kw),
        "greedy": lambda: ops.ntuple_greedy(b, w, STANDARD_4X6, action_dtype=torch.uint8, out=g_out, **kw),
        "td_update": lambda: ops.ntuple_td_update(b, target, w, STANDARD_4X6, alpha=1e-9, delta_out=delta, **kw),
        "tc_update": lambda: ops.ntuple_tc_update(b, target, w, c, acc, STANDARD_4X6, alpha=1e-9, delta_out=delta, **kw),
        "expectimax1": lambda: ops.ntuple_expectimax(b, w, STANDARD_4X6, depth=1, action_dtype=torch.uint8, out=x_out, **kw),
    }


def time_kernels(boards: torch.Tensor, sizes, rounds: int) -> dict:
    n = ops.ntuple_num_weights(STANDARD_4X6)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(0)
    nets = {}
    for stages in ((), TIMED_STAGES, ONE_TABLE_STAGES):
        s = len(stages) + 1
        w = torch.randn(s * n, device="cuda", generator=gen) * 10
        c = torch.rand((s * n, 2), device="cuda", generator=gen)
        nets[stages] = (w, c, torch.zeros((s * n, 2), device="cuda"))
    out = {}
    for lg in sizes:
        m = 1 << lg
        b = boards[:m]
        say(f"M=2^{lg}: stage shares of the boards under {TIMED_STAGES}: "
            + ", ".join(f"{x:.3f}" for x in stage_shares(b, TIMED_STAGES)))
        fns = {stages: op_fns(b, stages, *nets[stages]) for stages in nets}
        row = {}
        for op in fns[()]:
            iters = max(3, min(200, (1 << 24) // m)) if op == "expectimax1" else max(10, min(400, (1 << 27) // (m * 8)))
            runs = {(): [], TIMED_STAGES: [], ONE_TABLE_STAGES: []}
            for _ in range(rounds):
                for stages in runs:
                    runs[stages].append(min(time_graph(fns[stages][op], iters, repeats=1)))
            s1, s3, s2 = min(runs[()]), min(runs[TIMED_STAGES]), min(runs[ONE_TABLE_STAGES])
            row[op] = {"s1_us": runs[()], "s3_us": runs[TIMED_STAGES], "ratio": s3 / s1, "s2_one_table_us": runs[ONE_TABLE_STAGES],
                       "one_table_ratio": s2 / s1, "iters": iters}
            say(f"  {op:12s} S=1 {s1:9.1f} us  S=3 {s3:9.1f} us  ratio {s3 / s1:.3f}  "
                f"(rounds S=1 {min(runs[()]):.1f}-{max(runs[()]):.1f}, S=3 {min(runs[TIMED_STAGES]):.1f}-{max(runs[TIMED_STAGES]):.1f})"
                f"  | S=2 all in stage 0 {s2:9.1f} us  ratio {s2 / s1:.3f}")
        out[lg] = row
    for stages, (w, c, acc) in nets.items():
        assert not bool(acc.view(torch.int32).any()), "the TC accumulator is not all zero"
    return out


def fmt(p: dict) -> str:
    return f"mean score {p['mean_score']:.0f} p1024 {p['p1024']:.3f} p2048 {p['p2048']:.4f} ({p['seconds']} s)"


def at_time(points: list, t: float):
    done = [p for p in points if p["seconds"] <= t]
    return done[-1] if done else None


def main() -> None:
    p = argparse.ArgumentParser()
    p.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    p.add_argument("--quick", action="store_true", help="small sizes and few steps (a rehearsal, not a measurement)")
    args = p.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    q = args.quick
    res = {"device": device_info(), "tuples": STANDARD_4X6, "timed_stages": TIMED_STAGES}
    say(json.dumps(res["device"]))
    t_start = time.perf_counter()

    sizes = [12, 14] if q else [16, 18, 20]
    boards = steady_boards(1 << max(sizes))
    res["kernels"] = time_kernels(boards, sizes, 2 if q else 5)
    del boards
    torch.cuda.empty_cache()

    m = 1 << (10 if q else 14)
    steps = 4000 if q else 200000
    alpha = DEFAULT_ALPHA_TIMES_GAMES / m
    res["learning"] = {"m": m, "steps": steps, "alpha_times_games": DEFAULT_ALPHA_TIMES_GAMES, "seed": 0, "runs": {}}
    curves = {}
    for stages in ((), (10,), (11,)):
        _, curve = learner_run(m, alpha, steps, curve_every=steps // 10, net=NTupleNetwork(stages=stages))
        curves[stages] = curve
        res["learning"]["runs"][f"td0 stages={list(stages)}"] = curve
        say(f"td0 stages={stages}: final window {fmt(curve[-1])}, finite {curve[-1]['weights_finite']}")
    best = max(((10,), (11,)), key=lambda s: curves[s][-1]["mean_score"])
    _, lcurve = learner_run(m, alpha, steps, curve_every=steps // 10, net=NTupleNetwork(stages=best), horizon=3, lam=0.25)
    res["learning"]["runs"][f"td_lambda h=3 lam=0.25 stages={list(best)}"] = lcurve
    res["learning"]["better_split"] = list(best)
    say(f"better split by final mean score: {best}; TD(lambda) h=3 lambda=0.25 there: final window {fmt(lcurve[-1])}")
    base = curves[()]
    for name, curve in ((f"td0 {(10,)}", curves[(10,)]), (f"td0 {(11,)}", curves[(11,)]), (f"td_lambda {best}", lcurve)):
        say(f"curves: single-stage td0 against {name}")
        for a, b in zip(base, curve):
            same_t = at_time(base, b["seconds"])
            say(f"  step {a['step']}: S=1 {fmt(a)} | {name} {fmt(b)} | S=1 at {b['seconds']} s: "
                + (f"step {same_t['step']} mean score {same_t['mean_score']:.0f} p2048 {same_t['p2048']:.4f}" if same_t else "no window yet"))
    res["seconds"] = time.perf_counter() - t_start
    say(f"done in {res['seconds']:.0f} s")
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "stages_bench.json"), "w") as fh:
        fh.write(json.dumps(res, indent=1, default=float))
    with open(os.path.join(args.out_dir, "stages_bench.txt"), "w") as fh:
        fh.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
