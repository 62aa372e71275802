"""Temporal coherence (TC) learning of n-tuple networks (ops.ntuple_tc_update, TDAfterstateLearner(rule="tc")) against TD(0):
update time, learner step time, a TC step-size sweep and side-by-side learning curves.

    python tools/tc_bench.py [--out-dir DIR] [--quick]

- Learner step time: TDAfterstateLearner.step() with rule "td0" and "tc" at M = 4096, 2^14 and 2^16 (host clock around
  synchronised batches of 500 steps, 3 batches, default step sizes).
- Step-size sweep for TC: alpha = c / M for c = 0.1 ... 6.4 at M = 4096, 2^14 and 2^16, 30 000 steps each, the mean score and
  512 / 1024 shares of the episodes that end in the last quarter (tools/ntuple_bench.py's learner_run, the same columns as
  its TD(0) sweep).  The best c by mean score summed over the three sizes is the one the curves below use.
- Learning curves: 200 000 steps at M = 2^14 from zero weights, TC at the best c of the sweep next to TD(0) at its default,
  the same seed, in windows of 20 000 steps.
- Update time: tc_update against td_update on the same boards (a steady-state rollout of the in-kernel random policy, 400
  steps with auto-reset, at the largest size; smaller sizes take a prefix), the standard 4x6 network with zero weights and
  with the TC curve's trained weights and coherence, M = 2^16 ... 2^24, CUDA-graph timed (ntuple_bench's time_graph).
- Torch composition of the same definition up to 2^22 (index tensor, index_add_ into the accumulator, the apply over the
  unique entries): speed ratio, and a cross-check on 2^16 boards of delta (within fp32 summation-order tolerance: torch sums
  the 32 lookups in another order) and of the weights and coherence from the kernel's delta (within the float32 rounding
  bound of the atomics).
- The apply kernel without the plain load before the exchange (the library rebuilt with -DML2048_TC_APPLY_ALWAYS_EXCHANGE
  in a temporary directory, timed in a child process on the same boards and weights).
Device name and power limit are read in the same run.  Writes tc_bench.{json,txt} under --out-dir (default profiles/).
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch

from ntuple_bench import TorchComposed, device_info, learner_run, time_eager, time_graph

import ml2048_b200
from ml2048_b200 import ops
from ml2048_b200.build import COMPRESSIBLE_SRC, HOST_SRC, HOST_UNPACK_SRC, NVCC_FLAGS, SRC, nvcc_path
from ml2048_b200.ntuple import DEFAULT_ALPHA_TIMES_GAMES, STANDARD_4X6, NTupleNetwork, TDAfterstateLearner, default_alpha

LINES: list = []


def say(msg: str) -> None:
    LINES.append(msg)
    print(msg, flush=True)


class TorchTC(TorchComposed):
    """the TC update composed from torch ops: index tensor, index_add_ into the accumulator, apply over unique entries"""

    def tc_update(self, after, target, alpha, coh, acc, delta=None):
        idx = self.index(after)
        if delta is None:
            delta = alpha * (target - self.w[idx].sum(-1))
        flat = idx.reshape(-1)
        d = delta[:, None].expand_as(idx).reshape(-1)
        acc.index_add_(0, flat, torch.stack([d, d.abs()], dim=1))
        u = torch.unique(flat)
        da = acc[u, 1]
        u = u[da != 0]
        de, da = acc[u, 0], acc[u, 1]
        e0, a0 = coh[u, 0], coh[u, 1]
        beta = torch.where(a0 == 0, torch.ones_like(a0), e0.abs() / a0)
        self.w[u] += beta * de
        coh[u, 0] = e0 + de
        coh[u, 1] = a0 + da
        acc.zero_()
        return delta


def steady_boards(m: int) -> torch.Tensor:
    env = ml2048_b200.VecGame(m, output="torch", sync_free=True, track_merged=False)
    env.reset(0)
    for _ in range(400):
        env.step_random(auto_reset=True)
    torch.cuda.synchronize()
    b = env.observations()[0].clone()
    del env
    return b


def time_updates(boards, weights, coherence, sizes, iters) -> dict:
    """us per call of tc_update (and td_update) at each size, on copies of the weights"""
    out = {}
    for lg in sizes:
        m = 1 << lg
        b = boards[:m]
        target = torch.ones(m, device="cuda")  # non-zero deltas: an all-zero batch would skip the apply
        delta = torch.empty(m, device="cuda")
        w, c = weights.clone(), coherence.clone()
        acc = torch.zeros_like(c)
        out[lg] = {"tc_update": time_graph(lambda: ops.ntuple_tc_update(b, target, w, c, acc, STANDARD_4X6, alpha=1e-9,
                                                                        delta_out=delta), iters(m))}
        out[lg]["accum_zero_after"] = not bool(acc.view(torch.int32).any())
        del w, c, acc
    return out


def child_main(path: str) -> None:
    d = torch.load(path)
    boards, weights, coh = d["boards"].cuda(), d["weights"].cuda(), d["coherence"].cuda()
    res = time_updates(boards, weights, coh, d["sizes"], lambda m: max(3, min(200, (1 << 26) // (m * 8))))
    print(json.dumps(res))


def variant(tmp: str, boards, weights, coh, sizes) -> dict:
    so = os.path.join(tmp, "libml2048_b200_always_exchange.so")
    subprocess.run([nvcc_path(), *NVCC_FLAGS, "-DML2048_TC_APPLY_ALWAYS_EXCHANGE", "-o", so, SRC, HOST_SRC, HOST_UNPACK_SRC,
                    COMPRESSIBLE_SRC], check=True)
    path = os.path.join(tmp, "variant_inputs.pt")
    torch.save({"boards": boards.cpu(), "weights": weights.cpu(), "coherence": coh.cpu(), "sizes": sizes}, path)
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path], env=dict(os.environ, ML2048_LIB=so),
                         capture_output=True, text=True, check=True)
    return json.loads(out.stdout.strip().splitlines()[-1])


def cross_check(net_w, net_c, b) -> dict:
    """kernel against the torch composition on the same boards: delta within the value tolerance, weights and coherence from
    the kernel's delta within the float32 rounding bound (k + 2 roundings for w, k for E and A; k = adds to the entry)"""
    m = b.shape[0]
    target = torch.randn(m, device="cuda") * 1000
    alpha = 1e-3
    w_k, c_k = net_w.clone(), net_c.clone()
    acc = torch.zeros_like(c_k)
    d_k = ops.ntuple_tc_update(b, target, w_k, c_k, acc, STANDARD_4X6, alpha=alpha)
    tt = TorchTC(STANDARD_4X6, net_w.clone())
    idx = tt.index(b)
    d_t = alpha * (target - net_w[idx].sum(-1))
    tol_d = alpha * 64 * 2.0 ** -24 * (net_w[idx].abs().sum(-1) + target.abs())
    c_t = net_c.clone()
    tt.tc_update(b, target, alpha, c_t, torch.zeros_like(c_t), delta=d_k)
    flat = idx.reshape(-1)
    adds = torch.bincount(flat, minlength=net_w.numel()).double()
    sabs = torch.zeros(net_w.numel(), dtype=torch.float64, device="cuda").index_add_(
        0, flat, d_k.double().abs()[:, None].expand_as(idx).reshape(-1))
    a0 = net_c[:, 1].double()
    beta = torch.where(a0 == 0, torch.ones_like(a0), net_c[:, 0].double().abs() / a0)
    u = 2.0 ** -24
    # both sides are within the bound of the exact result: their difference within twice the bound
    bw = 2 * (adds + 2) * u * (net_w.double().abs() + beta * sabs)
    be = 2 * adds * u * (net_c[:, 0].double().abs() + sabs)
    ba = 2 * adds * u * (net_c[:, 1].double().abs() + sabs)
    return {"delta_within_tol": bool(((d_k - d_t).abs() <= tol_d).all()),
            "delta_max_abs_diff": float((d_k - d_t).abs().max()),
            "weights_within_bound": bool(((w_k.double() - tt.w.double()).abs() <= bw).all()),
            "E_within_bound": bool(((c_k[:, 0].double() - c_t[:, 0].double()).abs() <= be).all()),
            "A_within_bound": bool(((c_k[:, 1].double() - c_t[:, 1].double()).abs() <= ba).all()),
            "untouched_identical": bool(torch.equal(w_k[adds == 0], net_w[adds == 0]) and torch.equal(c_k[adds == 0], net_c[adds == 0])),
            "accum_zero_after": not bool(acc.view(torch.int32).any())}


def main() -> None:
    p = argparse.ArgumentParser()
    p.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    p.add_argument("--quick", action="store_true", help="small sizes and few steps (a rehearsal, not a measurement)")
    p.add_argument("--child", default=None, help=argparse.SUPPRESS)
    args = p.parse_args()
    if args.child:
        child_main(args.child)
        return
    assert torch.cuda.is_available(), "needs a GPU"
    q = args.quick
    res = {"device": device_info(), "tuples": STANDARD_4X6, "td0_alpha_times_games": DEFAULT_ALPHA_TIMES_GAMES}
    say(json.dumps(res["device"]))
    t_start = time.perf_counter()

    # learner step time
    res["learner_step_us"] = {}
    for m in ((4096,) if q else (4096, 1 << 14, 1 << 16)):
        row = {}
        for rule in ("td0", "tc"):
            env = ml2048_b200.VecGame(m, output="torch", sync_free=True, rng_mode="philox")
            learner = TDAfterstateLearner(env, NTupleNetwork(), rule=rule)
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
            row[rule] = reps
            del learner, env
        res["learner_step_us"][m] = row
        say(f"learner step M={m}: td0 {min(row['td0']):.1f} us, tc {min(row['tc']):.1f} us")

    # TC step-size sweep
    cs = (0.1, 0.2, 0.4, 0.8, 1.6, 3.2, 6.4)
    sweep_steps = 2000 if q else 30000
    res["tc_sweep"] = {}
    score = {c: 0.0 for c in cs}
    for m in ((4096,) if q else (4096, 1 << 14, 1 << 16)):
        for c in cs:
            _, curve = learner_run(m, c / m, sweep_steps, rule="tc")
            res["tc_sweep"][f"{m}/{c}"] = curve
            last = curve[-1]
            score[c] += last["mean_score"]
            say(f"tc sweep M={m} alpha*M={c} alpha={c / m:.3g}: last quarter {last['episodes']} episodes, mean score "
                f"{last['mean_score']:.0f}, p512 {last['p512']:.3f} p1024 {last['p1024']:.3f}, finite {last['weights_finite']}")
    best = max(cs, key=lambda c: score[c])
    res["tc_best_alpha_times_games"] = best
    say(f"tc sweep best alpha*M (mean score summed over the sizes): {best}")

    # learning curves, the same seed
    m = 1 << 14
    curve_steps = 20000 if q else 200000
    res["curves"] = {"m": m, "steps": curve_steps}
    nets = {}
    for rule, alpha in (("td0", default_alpha(m)), ("tc", best / m)):
        net, curve = learner_run(m, alpha, curve_steps, curve_every=curve_steps // 10, rule=rule)
        nets[rule] = net
        res["curves"][rule] = {"alpha": alpha, "points": curve}
    for a, b in zip(res["curves"]["td0"]["points"], res["curves"]["tc"]["points"]):
        say(f"curve step {a['step']}: td0 mean score {a['mean_score']:.0f} p512 {a['p512']:.3f} p1024 {a['p1024']:.3f} "
            f"p2048 {a['p2048']:.4f} ({a['seconds']} s) | tc mean score {b['mean_score']:.0f} p512 {b['p512']:.3f} "
            f"p1024 {b['p1024']:.3f} p2048 {b['p2048']:.4f} ({b['seconds']} s)")

    # update time
    sizes = [16, 18] if q else [16, 18, 20, 22, 24]
    boards = steady_boards(1 << max(sizes))
    zero_w = torch.zeros(ops.ntuple_num_weights(STANDARD_4X6), device="cuda")
    zero_c = torch.zeros((zero_w.numel(), 2), device="cuda")
    trained = nets["tc"]
    res["update"] = {}
    iters = lambda m: max(3, min(200, (1 << 26) // (m * 8)))  # noqa: E731
    torch_max = 18 if q else 22
    for wname, w, c in (("zero", zero_w, zero_c), ("trained", trained.weights, trained.coherence)):
        tc = time_updates(boards, w, c, sizes, iters)
        for lg in sizes:
            mm = 1 << lg
            b = boards[:mm]
            target = torch.ones(mm, device="cuda")
            delta = torch.empty(mm, device="cuda")
            w_td = w.clone()
            row = tc[lg]
            row["td_update"] = time_graph(lambda: ops.ntuple_td_update(b, target, w_td, STANDARD_4X6, alpha=1e-9, delta_out=delta),
                                          iters(mm))
            del w_td
            if lg <= torch_max:
                tt = TorchTC(STANDARD_4X6, w.clone())
                c_t = c.clone()
                acc_t = torch.zeros_like(c_t)
                row["torch_tc_update"] = time_eager(lambda: tt.tc_update(b, target, 1e-9, c_t, acc_t), 3)
                del tt, c_t, acc_t
            ratio = min(row["tc_update"]) / min(row["td_update"])
            line = f"{wname} M=2^{lg}: tc_update {min(row['tc_update']):.1f} us, td_update {min(row['td_update']):.1f} us, ratio {ratio:.2f}"
            if "torch_tc_update" in row:
                line += f", torch {min(row['torch_tc_update']):.1f} us ({min(row['torch_tc_update']) / min(row['tc_update']):.1f}x)"
            say(line + f", accumulator zero after {row['accum_zero_after']}")
        res["update"][wname] = tc
    res["cross_check"] = {wname: cross_check(w, c, boards[:1 << 16])
                          for wname, w, c in (("zero", zero_w, zero_c), ("trained", trained.weights, trained.coherence))}
    say(f"cross-check against the torch composition, 2^16 boards: {json.dumps(res['cross_check'])}")
    with tempfile.TemporaryDirectory() as tmp:
        res["always_exchange"] = variant(tmp, boards, trained.weights, trained.coherence, sizes)
    for lg in sizes:
        a, s = min(res["always_exchange"][str(lg)]["tc_update"]), min(res["update"]["trained"][lg]["tc_update"])
        say(f"trained M=2^{lg}: apply with the plain load first {s:.1f} us, always exchange {a:.1f} us")
    res["seconds"] = time.perf_counter() - t_start
    say(f"done in {res['seconds']:.0f} s")
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "tc_bench.json"), "w") as fh:
        fh.write(json.dumps(res, indent=1, default=float))
    with open(os.path.join(args.out_dir, "tc_bench.txt"), "w") as fh:
        fh.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
