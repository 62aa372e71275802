"""Delayed TD(lambda) / TC(lambda) for n-tuple networks (ops.ntuple_td_lambda_update / ntuple_tc_lambda_update,
TDAfterstateLearner(horizon=h, lam=...)) against TD(0) and TC: update time, learner step time, a (lambda, h) sweep, a coarse
step-size sweep and learning curves at equal steps and at equal wall time.

    python tools/lambda_bench.py [--out-dir DIR] [--quick]

- Learner step time: TDAfterstateLearner.step() for rule "td0" and "tc" at h = 1 (TD(0) / TC), 2, 4, 8 (lambda = 0.5), M = 4096,
  2^14 and 2^16 (host clock around synchronised batches of 500 steps, 3 batches, after 50 warm-up steps).
- (lambda, h) sweep: 30 000 steps at M = 2^14 from zero weights, lambda in {0.25, 0.5, 0.75} x h in {2, 3, 5} and h = 1, per
  rule at the rule's default alpha * M; the mean score and 512 / 1024 shares of the episodes that end in the last quarter
  (tools/ntuple_bench.py's learner_run, seed 0).  The best (lambda, h) of each rule by mean score is the one used below.
- A coarse alpha * M sweep at each rule's best (lambda, h): c in {0.25, 0.5, 2, 4} x the rule's default (the default itself
  is the sweep's run).
- Learning curves: 200 000 steps at M = 2^14, seed 0, windows of 20 000 steps (tc_bench.py's), each rule's best setting next
  to TD(0) and TC at their defaults; at equal steps, and at equal wall time (the baseline's window that ends last at or
  before each lambda window's time).
- Update time: td_lambda_update / tc_lambda_update at h = 1, 2, 4, 8 against td_update / tc_update on the same x_0 boards (a
  steady-state rollout of the in-kernel random policy, 400 steps with auto-reset at the largest size; smaller sizes take a
  prefix; slot s of the ring holds the boards rolled by s * 12 345 games), no end in any window (every value of the window is
  looked up), the standard 4x6 network with the weights (and coherence) the curves end with, M = 2^16 ... 2^24, CUDA-graph
  timed (ntuple_bench's time_graph).
Device name and power limit are read in the same run.  Writes lambda_bench.{json,txt} under --out-dir (default profiles/).
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
from ml2048_b200.ntuple import (DEFAULT_ALPHA_TIMES_GAMES, DEFAULT_TC_ALPHA_TIMES_GAMES, STANDARD_4X6, NTupleNetwork,
                                TDAfterstateLearner)

LINES: list = []
DEFAULT_C = {"td0": DEFAULT_ALPHA_TIMES_GAMES, "tc": DEFAULT_TC_ALPHA_TIMES_GAMES}


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


def learner_step_us(m: int, rule: str, h: int) -> list:
    env = ml2048_b200.VecGame(m, output="torch", sync_free=True, rng_mode="philox")
    learner = TDAfterstateLearner(env, NTupleNetwork(), rule=rule, horizon=h, lam=0.5)
    learner.reset(0)
    for _ in range(50):
        learner.step()
    torch.cuda.synchronize()
    reps = []
    for _ in range(3):
        t0 = time.perf_counter()
        for _ in range(500):
            learner.step()
        torch.cuda.synchronize()
        reps.append((time.perf_counter() - t0) / 500 * 1e6)
    del learner, env
    return reps


def fmt(p: dict) -> str:
    return f"mean score {p['mean_score']:.0f} p512 {p['p512']:.3f} p1024 {p['p1024']:.3f} p2048 {p['p2048']:.4f} ({p['seconds']} s)"


def at_time(points: list, t: float):
    """the window of `points` that ends last at or before t seconds (None before the first)"""
    done = [p for p in points if p["seconds"] <= t]
    return done[-1] if done else None


def time_updates(boards, nets, sizes, horizons, iters) -> dict:
    out = {}
    for lg in sizes:
        m = 1 << lg
        b = boards[:m]
        target = torch.ones(m, device="cuda")
        delta = torch.empty(m, device="cuda")
        row = {}
        for rule in ("td0", "tc"):
            net = nets[rule]
            w = net.weights.clone()
            c = net.coherence.clone() if rule == "tc" else None
            acc = torch.zeros_like(c) if rule == "tc" else None
            if rule == "tc":
                row["tc_update"] = time_graph(lambda: ops.ntuple_tc_update(b, target, w, c, acc, STANDARD_4X6, alpha=1e-9,
                                                                           delta_out=delta), iters(m))
            else:
                row["td_update"] = time_graph(lambda: ops.ntuple_td_update(b, target, w, STANDARD_4X6, alpha=1e-9, delta_out=delta),
                                              iters(m))
            for h in horizons:
                after = torch.stack([torch.roll(b, 12345 * s, 0) for s in range(h + 1)])
                reward = torch.full((h + 1, m), 4.0, device="cuda")
                ended = torch.zeros((h + 1, m), dtype=torch.uint8, device="cuda")
                newest = h - 1  # x_0 in slot h: the boards rolled by 12 345 * h
                if rule == "tc":
                    fn = lambda: ops.ntuple_tc_lambda_update(after, reward, ended, newest, w, c, acc, STANDARD_4X6,  # noqa: E731
                                                             alpha=1e-9, lam=0.5, delta_out=delta)
                else:
                    fn = lambda: ops.ntuple_td_lambda_update(after, reward, ended, newest, w, STANDARD_4X6, alpha=1e-9,  # noqa: E731
                                                             lam=0.5, delta_out=delta)
                row[f"{rule}_lambda_h{h}"] = time_graph(fn, iters(m))
                del after, reward, ended
            if rule == "tc":
                row["accum_zero_after"] = not bool(acc.view(torch.int32).any())
            del w, c, acc
        out[lg] = row
        base = {"td0": min(row["td_update"]), "tc": min(row["tc_update"])}
        for rule, name in (("td0", "td_update"), ("tc", "tc_update")):
            say(f"M=2^{lg} {name} {base[rule]:.1f} us | " + ", ".join(
                f"h={h} {min(row[f'{rule}_lambda_h{h}']):.1f} us ({min(row[f'{rule}_lambda_h{h}']) / base[rule]:.2f}x)" for h in horizons))
    return out


def main() -> None:
    p = argparse.ArgumentParser()
    p.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    p.add_argument("--quick", action="store_true", help="small sizes and few steps (a rehearsal, not a measurement)")
    args = p.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    q = args.quick
    res = {"device": device_info(), "tuples": STANDARD_4X6, "default_alpha_times_games": DEFAULT_C}
    say(json.dumps(res["device"]))
    t_start = time.perf_counter()
    horizons = (1, 2, 4, 8)

    # learner step time
    res["learner_step_us"] = {}
    for m in ((4096,) if q else (4096, 1 << 14, 1 << 16)):
        row = {f"{rule}/h{h}": learner_step_us(m, rule, h) for rule in ("td0", "tc") for h in horizons}
        res["learner_step_us"][m] = row
        say(f"learner step M={m}: " + ", ".join(f"{k} {min(v):.1f} us" for k, v in row.items()))

    # (lambda, h) sweep at each rule's default step size
    m = 1 << 14
    sweep_steps = 2000 if q else 30000
    settings = [(1, 0.5)] + [(h, lam) for h in (2, 3, 5) for lam in (0.25, 0.5, 0.75)]
    res["sweep"] = {}
    best = {}
    for rule in ("td0", "tc"):
        scores = {}
        for h, lam in settings:
            _, curve = learner_run(m, DEFAULT_C[rule] / m, sweep_steps, rule=rule, horizon=h, lam=lam)
            last = curve[-1]
            res["sweep"][f"{rule}/h{h}/lam{lam}"] = curve
            scores[(h, lam)] = last["mean_score"]
            say(f"sweep {rule} h={h} lambda={lam} alpha*M={DEFAULT_C[rule]}: last quarter {last['episodes']} episodes, mean score "
                f"{last['mean_score']:.0f}, p512 {last['p512']:.3f} p1024 {last['p1024']:.3f}, finite {last['weights_finite']}")
        best[rule] = max((s for s in settings if s[0] > 1), key=lambda s: scores[s])
        say(f"sweep {rule}: best (h, lambda) {best[rule]} mean score {scores[best[rule]]:.0f} against h=1 {scores[(1, 0.5)]:.0f}")
        # coarse step-size sweep at the best (lambda, h)
        h, lam = best[rule]
        cs = {DEFAULT_C[rule]: scores[best[rule]]}
        for f in (0.25, 0.5, 2.0, 4.0):
            c = DEFAULT_C[rule] * f
            _, curve = learner_run(m, c / m, sweep_steps, rule=rule, horizon=h, lam=lam)
            last = curve[-1]
            res["sweep"][f"{rule}/h{h}/lam{lam}/c{c}"] = curve
            cs[c] = last["mean_score"]
            say(f"alpha sweep {rule} h={h} lambda={lam} alpha*M={c}: mean score {last['mean_score']:.0f}, p512 {last['p512']:.3f} "
                f"p1024 {last['p1024']:.3f}, finite {last['weights_finite']}")
        bc = max(cs, key=lambda c: cs[c])
        best[rule] = (h, lam, bc)
        say(f"alpha sweep {rule}: best alpha*M {bc} (default {DEFAULT_C[rule]})")
    res["best"] = {rule: {"horizon": v[0], "lam": v[1], "alpha_times_games": v[2]} for rule, v in best.items()}

    # learning curves, the same seed
    curve_steps = 20000 if q else 200000
    res["curves"] = {"m": m, "steps": curve_steps}
    nets = {}
    for rule in ("td0", "tc"):
        h, lam, c = best[rule]
        net, base = learner_run(m, DEFAULT_C[rule] / m, curve_steps, curve_every=curve_steps // 10, rule=rule)
        _, lcurve = learner_run(m, c / m, curve_steps, curve_every=curve_steps // 10, rule=rule, horizon=h, lam=lam)
        nets[rule] = net
        res["curves"][rule] = {"baseline": {"alpha_times_games": DEFAULT_C[rule], "points": base},
                               "lambda": {"horizon": h, "lam": lam, "alpha_times_games": c, "points": lcurve}}
        say(f"curves {rule}: h=1 at alpha*M={DEFAULT_C[rule]} against h={h} lambda={lam} alpha*M={c}")
        for a, b in zip(base, lcurve):
            same_t = at_time(base, b["seconds"])
            say(f"  step {a['step']}: h=1 {fmt(a)} | lambda {fmt(b)} | h=1 at {b['seconds']} s: "
                + (f"step {same_t['step']} mean score {same_t['mean_score']:.0f}" if same_t else "no window yet"))

    # update time
    sizes = [16, 18] if q else [16, 18, 20, 22, 24]
    boards = steady_boards(1 << max(sizes))
    iters = lambda m: max(3, min(200, (1 << 26) // (m * 8)))  # noqa: E731
    res["update"] = time_updates(boards, nets, sizes, horizons, iters)
    res["seconds"] = time.perf_counter() - t_start
    say(f"done in {res['seconds']:.0f} s")
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "lambda_bench.json"), "w") as fh:
        fh.write(json.dumps(res, indent=1, default=float))
    with open(os.path.join(args.out_dir, "lambda_bench.txt"), "w") as fh:
        fh.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
