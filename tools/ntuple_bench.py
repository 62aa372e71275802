"""N-tuple network kernels (ops.ntuple_value / ntuple_greedy / ntuple_td_update) against their ceilings, the same operations
composed from torch ops, TDAfterstateLearner step time, a step-size sweep and a learning curve.

    python tools/ntuple_bench.py [--sizes 16,18,20,22,24] [--out-dir DIR]

- Boards: a steady-state rollout of the in-kernel random policy (auto-reset fused in, 400 steps) at the largest size; smaller
  sizes take a prefix.  The standard 4x6 network (256 MiB of weights, more than the 126 MB L2).
- Kernels: `iters` back-to-back launches in one CUDA graph, CUDA-event time over `iters`, 3 replays; with zero weights and
  with the weights the learning curve below ends with (the index distribution, and with it the L2 hit rate, follows play).
- Ceilings in the same run: a bare random 4-byte gather (tools/gather_ceiling.cu, hashed uniform indices) over a 256 MiB
  table and over an L2-resident 16 MiB table; a device-to-device copy for the byte floor of each kernel's own reads and writes.
  Lookups: greedy 128 per board (4 directions x 4 tuples x 8 images; fewer where a direction is invalid), value 32, the
  update 32 reads + 32 atomics per game.
- Torch-composed comparison: ops.afterstates + an index tensor + gather / sum / argmax, and index_put_(accumulate=True),
  checked against the kernels on the same boards (values within fp32 summation-order tolerance, actions where the best q
  leads by more than that).
- TDAfterstateLearner.step() at M = 4096 and 2^16 (host clock around synchronised batches of steps); a step-size sweep
  alpha = c / M at M = 4096, 2^14 and 2^16 (fixed steps each, mean score of the episodes that end in the last quarter); a
  learning curve at M = 2^14 with the default step size.
Device name and power limit are read in the same run.
"""

from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import ml2048_b200
from ml2048_b200 import ops
from ml2048_b200.build import nvcc_path
from ml2048_b200.ntuple import DEFAULT_ALPHA_TIMES_GAMES, STANDARD_4X6, NTupleNetwork, TDAfterstateLearner, default_alpha


def device_info() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        q = "unknown"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def time_graph(fn, iters: int, repeats: int = 3) -> list[float]:
    """us per call of `fn` over `iters` calls captured back to back in one CUDA graph"""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
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


def time_eager(fn, iters: int, repeats: int = 3) -> list[float]:
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(repeats):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(iters):
            fn()
        t1.record()
        t1.synchronize()
        out.append(t0.elapsed_time(t1) * 1e3 / iters)
    return out


def copy_gbs() -> float:
    a = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    us = min(time_eager(lambda: b.copy_(a), 20))
    del a, b
    return 2 * (1 << 31) / us / 1e3  # read + write, GB/s


def gather_ceiling(tmp: str) -> dict:
    so = os.path.join(tmp, "libgather_ceiling.so")
    subprocess.run([nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-shared", "-Xcompiler", "-fPIC", "-o", so,
                    os.path.join(ROOT, "tools", "gather_ceiling.cu")], check=True)
    lib = ctypes.CDLL(so)
    lib.gather_ceiling.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    res = {}
    threads, lookups = 1 << 22, 32
    out = torch.empty(threads, dtype=torch.float32, device="cuda")
    for name, log2 in (("256MiB", 26), ("16MiB_L2", 22)):
        table = torch.rand(1 << log2, device="cuda")
        us = time_graph(lambda: lib.gather_ceiling(table.data_ptr(), log2, lookups, out.data_ptr(), threads,
                                                   torch.cuda.current_stream().cuda_stream), 50)
        res[name] = {"us": us, "lookups_per_s": threads * lookups / (min(us) * 1e-6)}
        del table
    return res


class TorchComposed:
    """value / greedy / td_update of the network composed from torch ops (the comparison line)"""

    def __init__(self, tuples, weights):
        sym = []
        for g in range(8):
            sym.append([4 * (f[0]) + f[1] for f in [self._src(g, c) for c in range(16)]])
        self.w = weights
        src, shift, offs = [], [], []
        off = 0
        for t in tuples:
            for g in range(8):
                src.append([sym[g][c] for c in t] + [0] * (6 - len(t)))
                shift.append([4 * j for j in range(len(t))] + [63] * (6 - len(t)))
                offs.append(off)
            off += 16 ** len(t)
        self.src = torch.tensor(src, device="cuda")              # (8K, 6)
        self.shift = torch.tensor(shift, device="cuda")          # (8K, 6); 63 = a padding column that must add 0
        self.valid_col = (self.shift < 63)
        self.offs = torch.tensor(offs, device="cuda")

    @staticmethod
    def _src(g, cell):
        r, c = divmod(cell, 4)
        return [(r, c), (r, 3 - c), (3 - r, c), (3 - r, 3 - c), (c, r), (c, 3 - r), (3 - c, r), (3 - c, 3 - r)][g]

    def index(self, boards):  # (..., 16) -> (..., 8K) int64
        cells = boards.long().clamp_(max=15)[..., self.src]       # (..., 8K, 6)
        shift = torch.where(self.valid_col, self.shift, 0)
        return ((cells << shift) * self.valid_col).sum(-1) + self.offs

    def value(self, boards):
        return self.w[self.index(boards)].sum(-1)

    def greedy(self, boards, reward_fn=None):
        a = ops.afterstates(boards, reward_fn=reward_fn)
        v = self.value(a["state"])
        q = torch.where(a["valid_actions"].bool(), a["reward"] + v, float("-inf"))
        act = q.argmax(dim=1)
        return act, q

    def td_update(self, after, target, alpha):
        idx = self.index(after)
        delta = alpha * (target - self.w[idx].sum(-1))
        self.w.index_put_((idx.reshape(-1),), delta[:, None].expand_as(idx).reshape(-1), accumulate=True)
        return delta


def learner_run(m: int, alpha: float, steps: int, seed: int = 0, curve_every: int = 0, net=None, rule: str = "td0",
                horizon: int = 1, lam: float = 0.5):
    net = net or NTupleNetwork()
    env = ml2048_b200.VecGame(m, output="torch", sync_free=True, rng_mode="philox")
    learner = TDAfterstateLearner(env, net, alpha=alpha, rule=rule, horizon=horizon, lam=lam)
    learner.reset(seed)
    curve, t0 = [], time.perf_counter()
    window = curve_every or max(steps // 4, 1)
    for i in range(steps):
        learner.step()
        if (i + 1) % window == 0 or i + 1 == steps:
            st = env.episode_stats(reset=True)
            eps = max(st["episodes"], 1)
            h = st["max_tile_hist"]
            curve.append({"step": i + 1, "seconds": round(time.perf_counter() - t0, 2), "episodes": st["episodes"],
                          "mean_score": st["score_sum"] / eps, "mean_steps": st["step_sum"] / eps,
                          "p512": float(h[9:].sum() / eps), "p1024": float(h[10:].sum() / eps), "p2048": float(h[11:].sum() / eps),
                          "weights_finite": bool(torch.isfinite(net.weights).all())})
    return net, curve


def main() -> None:
    p = argparse.ArgumentParser()
    p.add_argument("--sizes", default="16,18,20,22,24")
    p.add_argument("--torch-max", type=int, default=22, help="largest log2 M of the torch-composed comparison")
    p.add_argument("--sweep-steps", type=int, default=30000)
    p.add_argument("--curve-steps", type=int, default=200000)
    p.add_argument("--alpha-times-games", default="0.1,0.2,0.4,0.8,1.6,3.2", help="the swept alpha * M")
    p.add_argument("--out-dir", default=None)
    args = p.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    sizes = [int(x) for x in args.sizes.split(",")]
    res = {"device": device_info(), "tuples": STANDARD_4X6, "default_alpha_times_games": DEFAULT_ALPHA_TIMES_GAMES}
    print(json.dumps(res["device"]), flush=True)

    # learner step time, step-size sweep and the learning curve (its weights are the "trained" weights below)
    res["learner_step_us"] = {}
    for m in (4096, 1 << 16):
        net = NTupleNetwork()
        env = ml2048_b200.VecGame(m, output="torch", sync_free=True, rng_mode="philox")
        learner = TDAfterstateLearner(env, net)
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
        res["learner_step_us"][m] = reps
        print(f"learner step M={m}: {min(reps):.1f} us", flush=True)
    res["alpha_sweep"] = {}
    for m in (4096, 1 << 14, 1 << 16):
        for c in (float(a) for a in args.alpha_times_games.split(",")):
            alpha = c / m
            _, curve = learner_run(m, alpha, args.sweep_steps)
            res["alpha_sweep"][f"{m}/{c}"] = curve
            last = curve[-1]
            print(f"sweep M={m} alpha*M={c} alpha={alpha:.3g}: last quarter {last['episodes']} episodes, mean score {last['mean_score']:.0f}, "
                  f"p512 {last['p512']:.3f} p1024 {last['p1024']:.3f}, finite {last['weights_finite']}", flush=True)
    trained, curve = learner_run(1 << 14, default_alpha(1 << 14), args.curve_steps, curve_every=args.curve_steps // 10)
    res["learning_curve"] = {"m": 1 << 14, "alpha": default_alpha(1 << 14), "points": curve}
    for c in curve:
        print(f"curve step {c['step']} ({c['seconds']} s): {c['episodes']} episodes, mean score {c['mean_score']:.0f}, "
              f"p512 {c['p512']:.3f} p1024 {c['p1024']:.3f} p2048 {c['p2048']:.4f}", flush=True)

    # ceilings
    with tempfile.TemporaryDirectory() as tmp:
        res["gather_ceiling"] = gather_ceiling(tmp)
    res["copy_gbs"] = copy_gbs()
    print(f"ceilings: gather 256 MiB {res['gather_ceiling']['256MiB']['lookups_per_s'] / 1e9:.1f} G/s, "
          f"L2 {res['gather_ceiling']['16MiB_L2']['lookups_per_s'] / 1e9:.1f} G/s, copy {res['copy_gbs']:.0f} GB/s", flush=True)

    # kernels
    mmax = 1 << max(sizes)
    env = ml2048_b200.VecGame(mmax, output="torch", sync_free=True, track_merged=False)
    env.reset(0)
    for _ in range(400):
        env.step_random(auto_reset=True)
    torch.cuda.synchronize()
    boards_all = env.observations()[0].clone()
    del env
    valid_share = float(ops.valid_actions(boards_all[:1 << 20]).float().mean())
    res["valid_direction_share"] = valid_share
    res["kernels"] = {}
    floor_bytes = {"value": 20, "greedy": 16 + 16 + 4 + 4 + 8, "td_update": (16 + 4 + 1 + 4) + (16 + 1 + 4)}
    lookups = {"value": 32, "greedy": 128 * valid_share, "td_update": 64}
    zero = NTupleNetwork()
    for wname, net in (("zero", zero), ("trained", trained)):
        for lg in sizes:
            m = 1 << lg
            b = boards_all[:m]
            iters = max(3, min(200, (1 << 26) // (m * 8)))
            out_v = torch.empty(m, device="cuda")
            g_out = {"action": torch.empty(m, dtype=torch.int64, device="cuda"), "state": torch.empty((m, 16), dtype=torch.uint8, device="cuda"),
                     "reward": torch.empty(m, device="cuda"), "value": torch.empty(m, device="cuda")}
            target = torch.zeros(m, device="cuda")
            delta = torch.empty(m, device="cuda")
            w_td = net.weights.clone()
            row = {}
            row["value"] = time_graph(lambda: ops.ntuple_value(b, net.weights, net.tuples, out=out_v), iters)
            row["greedy"] = time_graph(lambda: ops.ntuple_greedy(b, net.weights, net.tuples, out=g_out), iters)
            row["td_update"] = time_graph(lambda: ops.ntuple_td_update(b, target, w_td, net.tuples, alpha=1e-9, delta_out=delta), iters)
            for k in list(row):
                us = min(row[k])
                row[k] = {"us": row[k], "boards_per_s": m / (us * 1e-6), "lookups_per_s": m * lookups[k] / (us * 1e-6),
                          "vs_gather_256MiB": m * lookups[k] / (us * 1e-6) / res["gather_ceiling"]["256MiB"]["lookups_per_s"],
                          "byte_floor_us": m * floor_bytes[k] / (res["copy_gbs"] * 1e3)}
            if lg <= args.torch_max:
                tc = TorchComposed(net.tuples, net.weights.clone())
                row["torch_value"] = {"us": time_eager(lambda: tc.value(b), 3)}
                row["torch_greedy"] = {"us": time_eager(lambda: tc.greedy(b), 3)}
                tgt = torch.zeros(m, device="cuda")
                row["torch_td_update"] = {"us": time_eager(lambda: tc.td_update(b, tgt, 1e-9), 3)}
                # outputs against each other on a sample
                s = b[:1 << 16]
                tcs = TorchComposed(net.tuples, net.weights)
                v_k, v_t = ops.ntuple_value(s, net.weights, net.tuples), tcs.value(s)
                tol = 64 * 2.0 ** -24 * net.weights[tcs.index(s)].abs().sum(-1)  # two orders of 32 float32 adds, each within 31 u sum|w|
                gk = ops.ntuple_greedy(s, net.weights, net.tuples)
                act_t, q = TorchComposed(net.tuples, net.weights).greedy(s)
                top2 = q.topk(2, dim=1).values
                clear = (top2[:, 0] - top2[:, 1]) > 1e-4 * (top2[:, 0].abs() + 1)
                row["check"] = {"value_max_rel": float(((v_k - v_t).abs() / (v_t.abs() + 1)).max()),
                                "value_within_tol": bool(((v_k - v_t).abs() <= tol).all()),
                                "actions_equal_where_clear": bool((gk["action"][clear] == act_t[clear]).all()),
                                "clear_share": float(clear.float().mean())}
                del tc
            res["kernels"][f"{wname}/{m}"] = row
            line = " ".join(f"{k} {min(v['us']):.1f}us" for k, v in row.items() if isinstance(v, dict) and "us" in v)
            print(f"{wname} M=2^{lg}: {line} {row.get('check', '')}", flush=True)
            del w_td

    text = json.dumps(res, indent=1, default=float)
    if args.out_dir:
        os.makedirs(args.out_dir, exist_ok=True)
        with open(os.path.join(args.out_dir, "ntuple_bench.json"), "w") as fh:
            fh.write(text)
    print("done", flush=True)


if __name__ == "__main__":
    main()
