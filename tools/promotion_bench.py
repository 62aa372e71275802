"""Weight promotion of multi-stage n-tuple networks (the ``promoted=`` argument of ops.ntuple_*, NTupleNetwork(...,
promotion=True)): what promotion costs per kernel against the staged kernels without it, and how promoting networks learn.

    python tools/promotion_bench.py [--out-dir DIR] [--quick]

- Kernel cost: S = 3 with stages (6, 7), the standard 4x6 network with seeded random weights, promoting against not
  promoting, on stages_bench's steady-state boards at M = 2^16, 2^18 and 2^20.  ntuple_value, ntuple_greedy,
  ntuple_td_update, ntuple_tc_update and ntuple_expectimax (depth 1) are timed as CUDA-graph replays of back-to-back calls
  (ntuple_bench's time_graph), the two networks alternating, 5 rounds; the figure is the minimum over rounds and the ratio
  of the minima.  Promoting runs with every mark set (the steady state: the promote phase finds nothing to do); the reads
  run a second time with every mark clear (each lookup of a stage >= 1 board falls through to stage 0).  The promote phase
  that does promote is timed on td_update: before each call the marks are restored to all clear by a copy outside the
  timed region, CUDA events around each call, the minimum over calls.  Updates run with alpha = 1e-9 so that repeated
  calls leave the weights as they are up to rounding.
- Learning: M = 2^14, seed 0, 200 000 learner steps from zero weights, windows of 20 000 steps (ntuple_bench's
  learner_run), all in this process: TD(0) with one stage; TD(0) with stages (10,) and (11,), without and with promotion;
  TD(lambda) with h = 3, lambda = 0.25 with one stage and with promotion at the promoting split with the better final mean
  score.  At equal steps and at equal wall time (the single-stage window that ends last at or before each window's time).
  Every run uses the default step size, which was swept for single-stage networks only; other seeds are not run.
Device name and power limit are read in the same run.  Writes promotion_bench.{json,txt} under --out-dir (default
profiles/).
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
from stages_bench import at_time, fmt, op_fns, stage_shares, steady_boards

from ml2048_b200 import ops
from ml2048_b200.ntuple import DEFAULT_ALPHA_TIMES_GAMES, STANDARD_4X6, NTupleNetwork

LINES: list = []
TIMED_STAGES = (6, 7)


def say(msg: str) -> None:
    LINES.append(msg)
    print(msg, flush=True)


def with_marks(marks: torch.Tensor, b, w, c, acc) -> dict:
    """op_fns's calls with ``promoted=marks``"""
    m = b.shape[0]
    dev = b.device
    target = torch.ones(m, device=dev)
    delta = torch.empty(m, device=dev)
    value = torch.empty(m, device=dev)
    g_out = {"action": torch.empty(m, dtype=torch.uint8, device=dev), "state": torch.empty((m, 16), dtype=torch.uint8, device=dev),
             "reward": torch.empty(m, device=dev), "value": torch.empty(m, device=dev)}
    x_out = dict(g_out, q=torch.empty((m, 4), device=dev))
    kw = {"stages": TIMED_STAGES, "promoted": marks}
    return {
        "value": lambda: ops.ntuple_value(b, w, STANDARD_4X6, out=value, **kw),
        "greedy": lambda: ops.ntuple_greedy(b, w, STANDARD_4X6, action_dtype=torch.uint8, out=g_out, **kw),
        "td_update": lambda: ops.ntuple_td_update(b, target, w, STANDARD_4X6, alpha=1e-9, delta_out=delta, **kw),
        "tc_update": lambda: ops.ntuple_tc_update(b, target, w, c, acc, STANDARD_4X6, alpha=1e-9, delta_out=delta, **kw),
        "expectimax1": lambda: ops.ntuple_expectimax(b, w, STANDARD_4X6, depth=1, action_dtype=torch.uint8, out=x_out, **kw),
    }


def time_promoting_update(fn, marks: torch.Tensor, clear: torch.Tensor, calls: int) -> list:
    """us of each call of ``fn`` with the marks restored to ``clear`` before it, outside the timed region"""
    out = []
    for _ in range(calls):
        marks.copy_(clear)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        fn()
        t1.record()
        t1.synchronize()
        out.append(t0.elapsed_time(t1) * 1e3)
    return out


def time_kernels(boards: torch.Tensor, sizes, rounds: int) -> dict:
    n = ops.ntuple_num_weights(STANDARD_4X6)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(0)
    w = torch.randn(3 * n, device="cuda", generator=gen) * 10
    c = torch.rand((3 * n, 2), device="cuda", generator=gen)
    acc = torch.zeros((3 * n, 2), device="cuda")
    full = torch.full((n,), 3, dtype=torch.uint8, device="cuda")
    clear = torch.zeros((n,), dtype=torch.uint8, device="cuda")
    marks = full.clone()
    out = {}
    for lg in sizes:
        m = 1 << lg
        b = boards[:m]
        say(f"M=2^{lg}: stage shares of the boards under {TIMED_STAGES}: "
            + ", ".join(f"{x:.3f}" for x in stage_shares(b, TIMED_STAGES)))
        staged = op_fns(b, TIMED_STAGES, w, c, acc)
        promoting = with_marks(marks, b, w, c, acc)
        row = {}
        for op in staged:
            iters = max(3, min(200, (1 << 24) // m)) if op == "expectimax1" else max(10, min(400, (1 << 27) // (m * 8)))
            reads = op in ("value", "greedy", "expectimax1")
            runs = {"staged": [], "all_marks": [], "no_marks": []} if reads else {"staged": [], "all_marks": []}
            for _ in range(rounds):
                runs["staged"].append(min(time_graph(staged[op], iters, repeats=1)))
                marks.copy_(full)
                runs["all_marks"].append(min(time_graph(promoting[op], iters, repeats=1)))
                if reads:
                    marks.copy_(clear)
                    runs["no_marks"].append(min(time_graph(promoting[op], iters, repeats=1)))
            marks.copy_(full)
            base = min(runs["staged"])
            row[op] = {k + "_us": v for k, v in runs.items()}
            row[op]["iters"] = iters
            line = f"  {op:12s} staged {base:9.1f} us  promoting, all marks {min(runs['all_marks']):9.1f} us  ratio " \
                   f"{min(runs['all_marks']) / base:.3f}"
            row[op]["ratio_all_marks"] = min(runs["all_marks"]) / base
            if reads:
                row[op]["ratio_no_marks"] = min(runs["no_marks"]) / base
                line += f"  | no marks {min(runs['no_marks']):9.1f} us  ratio {min(runs['no_marks']) / base:.3f}"
            say(line)
        # the promote phase that promotes: td_update from all-clear marks, against the same call with all marks set
        fn = promoting["td_update"]
        fn()
        promo = time_promoting_update(fn, marks, clear, 3 * rounds)
        steady = time_promoting_update(fn, marks, full, 3 * rounds)
        row["td_update_promoting"] = {"clear_us": promo, "all_marks_us": steady, "ratio": min(promo) / min(steady)}
        say(f"  td_update one call: marks all clear (every stage >= 1 entry of the batch promoted) {min(promo):9.1f} us, "
            f"all marks set {min(steady):9.1f} us, ratio {min(promo) / min(steady):.3f}")
        marks.copy_(full)
        out[lg] = row
    assert not bool(acc.view(torch.int32).any()), "the TC accumulator is not all zero"
    return out


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
    for stages, promotion in (((), False), ((10,), False), ((10,), True), ((11,), False), ((11,), True)):
        net = NTupleNetwork(stages=stages, promotion=promotion)
        _, curve = learner_run(m, alpha, steps, curve_every=steps // 10, net=net)
        name = f"td0 stages={list(stages)}" + (" promotion" if promotion else "")
        curves[name] = curve
        res["learning"]["runs"][name] = curve
        extra = f", stage >= 1 entries written {int((net.promoted != 0).sum())}" if promotion else ""
        say(f"{name}: final window {fmt(curve[-1])}, finite {curve[-1]['weights_finite']}{extra}")
        del net
        torch.cuda.empty_cache()
    best = max(((10,), (11,)), key=lambda s: curves[f"td0 stages={list(s)} promotion"][-1]["mean_score"])
    res["learning"]["better_promoting_split"] = list(best)
    for stages, promotion in (((), False), (best, True)):
        name = f"td_lambda h=3 lam=0.25 stages={list(stages)}" + (" promotion" if promotion else "")
        _, curve = learner_run(m, alpha, steps, curve_every=steps // 10, net=NTupleNetwork(stages=stages, promotion=promotion),
                               horizon=3, lam=0.25)
        curves[name] = curve
        res["learning"]["runs"][name] = curve
        say(f"{name}: final window {fmt(curve[-1])}, finite {curve[-1]['weights_finite']}")
        torch.cuda.empty_cache()
    say(f"better promoting split by final mean score: {best}")
    for base_name in ("td0 stages=[]", "td_lambda h=3 lam=0.25 stages=[]"):
        base = curves[base_name]
        for name, curve in curves.items():
            if name == base_name or name.startswith("td0") != base_name.startswith("td0"):
                continue
            say(f"curves: {base_name} against {name}")
            for a, b in zip(base, curve):
                same_t = at_time(base, b["seconds"])
                say(f"  step {a['step']}: base {fmt(a)} | {fmt(b)} | base at {b['seconds']} s: "
                    + (f"step {same_t['step']} mean score {same_t['mean_score']:.0f} p2048 {same_t['p2048']:.4f}" if same_t
                       else "no window yet"))
    res["seconds"] = time.perf_counter() - t_start
    say(f"done in {res['seconds']:.0f} s")
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "promotion_bench.json"), "w") as fh:
        fh.write(json.dumps(res, indent=1, default=float))
    with open(os.path.join(args.out_dir, "promotion_bench.txt"), "w") as fh:
        fh.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
