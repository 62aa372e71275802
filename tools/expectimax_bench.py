"""Expectimax over an n-tuple network (ops.ntuple_expectimax): kernel time, work per board, the same search composed from
torch ops, the alternative depth-1 mapping, and play strength against the greedy move.

    python tools/expectimax_bench.py [--out-dir DIR] [--quick]

- Weights: the standard 4x6 network trained in this run with TDAfterstateLearner (M = 2^14, 100 000 steps, default alpha).
- Boards: steady-state boards of that network's own greedy play (M = 2^20 games, 1500 greedy steps with auto-reset); smaller
  sizes take a prefix.
- Kernel time: `iters` back-to-back launches in one CUDA graph, CUDA-event time over `iters`, 3 replays (tools/ntuple_bench.py's
  time_graph), for depth 1 at M = 2^12 ... 2^20 and depth 2 at M = 2^10 ... 2^14, two_prob 0.8, normal reward.  Against it:
  ntuple_greedy on the same boards, and the gather ceilings of tools/gather_ceiling.cu measured in the same run.
- Work per board: leaf evaluations (afterstates whose V the search reads) and table lookups (8 per tuple per leaf), counted
  exactly by enumerating each board's tree with ops.afterstates.
- Composed baseline: depth 1 from ops.afterstates + spawn enumeration in torch + ops.afterstates + ops.ntuple_value + torch
  reductions at M = 2^14, checked against the kernel (actions and value bits).
- Alternative mapping: the library rebuilt with -DML2048_EXPECTIMAX_WARP_PER_BOARD (one warp per board instead of one warp per
  (board, root direction)) times depth 1 on the same boards and weights in a child process; its outputs must equal the
  shipped kernel's bit for bit.
- Strength: greedy, depth 1 and depth 2 on the trained weights, every game played once from reset to its end (episode log),
  the same Philox seed for all three; mean score and length, the share reaching 2048 / 4096 / 8192 / 16384, wall time per move.
Device name and power limit are read in the same run.  Writes expectimax_bench.{json,txt} under --out-dir (default
profiles/).
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

import numpy as np
import torch

from ntuple_bench import device_info, gather_ceiling, time_eager, time_graph

import ml2048_b200
from ml2048_b200 import ops
from ml2048_b200.build import NVCC_FLAGS, nvcc_path, SRC, HOST_SRC, HOST_UNPACK_SRC, COMPRESSIBLE_SRC
from ml2048_b200.ntuple import STANDARD_4X6, NTupleNetwork, TDAfterstateLearner

TWO_PROB = 0.8
LOOKUPS_PER_LEAF = 8 * len(STANDARD_4X6)


def outs(m: int) -> dict:
    dev = "cuda"
    return {"action": torch.empty((m,), dtype=torch.uint8, device=dev), "state": torch.empty((m, 16), dtype=torch.uint8, device=dev),
            "reward": torch.empty((m,), dtype=torch.float32, device=dev), "value": torch.empty((m,), dtype=torch.float32, device=dev),
            "q": torch.empty((m, 4), dtype=torch.float32, device=dev)}


def time_depth1(boards, weights, sizes, iters) -> dict:
    res = {}
    for lg in sizes:
        m = 1 << lg
        b, o = boards[:m].contiguous(), outs(m)
        us = time_graph(lambda: ops.ntuple_expectimax(b, weights, STANDARD_4X6, depth=1, two_prob=TWO_PROB, action_dtype=torch.uint8, out=o),
                        iters(m))
        res[lg] = us
    return res


# ---- the search tree, enumerated with torch ops ------------------------------------------------------


def spawn_children(after: torch.Tensor, p2: float, p4: float):
    """every spawn outcome of (N,16) afterstates: children (N,16,T,16) with tile T_i in cell c, and keep (N,16,T), true where
    cell c is empty (T = the tiles of non-zero probability, 2 before 4)"""
    n = after.shape[0]
    empty = after == 0
    tiles = [t for t, p in ((1, p2), (2, p4)) if p > 0]
    child = after[:, None, None, :].expand(n, 16, len(tiles), 16).clone()
    eye = torch.eye(16, dtype=torch.uint8, device=after.device)
    for i, t in enumerate(tiles):
        child[:, :, i, :] += eye * t
    keep = empty[:, :, None].expand(n, 16, len(tiles))
    return child, keep


def tree_counts(boards: torch.Tensor, depth: int, kind="normal") -> int:
    """leaf evaluations (afterstates whose V is read) of all boards' trees at two_prob = TWO_PROB, counted exactly"""
    p2 = float(np.float32(TWO_PROB))
    p4 = float(np.float32(1) - np.float32(TWO_PROB))
    leaves = 0
    for i in range(0, boards.shape[0], 1 << 12):
        level = boards[i:i + (1 << 12)]
        for d in range(depth):
            a = ops.afterstates(level, reward_fn=kind)
            after = a["state"].reshape(-1, 16)[a["valid_actions"].reshape(-1).bool()]
            child, keep = spawn_children(after, p2, p4)
            level = child[keep].reshape(-1, 16).contiguous()
            if d == depth - 1:
                leaves += int(ops.afterstates(level, reward_fn=kind)["valid_actions"].sum())
    return leaves


def composed_depth1(boards: torch.Tensor, weights: torch.Tensor, kind="normal"):
    """depth-1 expectimax from existing ops and torch reductions, in the definition's arithmetic order"""
    p2 = torch.tensor(np.float32(TWO_PROB), device="cuda")
    p4 = torch.tensor(np.float32(1) - np.float32(TWO_PROB), device="cuda")
    m = boards.shape[0]
    a = ops.afterstates(boards, reward_fn=kind)
    after = a["state"].reshape(-1, 16)
    child, keep = spawn_children(after, TWO_PROB, 1 - TWO_PROB)                   # (4M,16,2,16), (4M,16,2)
    a2 = ops.afterstates(child[keep].contiguous(), reward_fn=kind)                 # the spawns into empty cells only
    v = ops.ntuple_value(a2["state"].reshape(-1, 16), weights, STANDARD_4X6).reshape(-1, 4)
    x = a2["reward"] + v
    valid2 = a2["valid_actions"].bool()
    key = torch.where(valid2 & ~torch.isnan(x), x, float("-inf"))
    mx = torch.zeros(keep.shape, dtype=torch.float32, device="cuda")
    mx[keep] = torch.where(valid2.any(1), key.max(1).values, 0.0)
    t = p2 * mx[..., 0] + p4 * mx[..., 1]                                          # separate multiply and add kernels: no FMA
    empty = keep[..., 0]
    s = torch.zeros(after.shape[0], dtype=torch.float32, device="cuda")
    started = torch.zeros(after.shape[0], dtype=torch.bool, device="cuda")
    for c in range(16):
        e = empty[:, c]
        s = torch.where(e, torch.where(started, s + t[:, c], t[:, c]), s)
        started |= e
    n = empty.sum(1).clamp(min=1).float()
    e_val = (s / n).reshape(m, 4)
    valid = a["valid_actions"].bool()
    q = torch.where(valid, a["reward"] + e_val, float("-inf"))
    qk = torch.where(torch.isnan(q), float("-inf"), q)
    act = torch.where(valid.any(1), qk.argmax(1), 0)
    return act, torch.where(valid.any(1), e_val.gather(1, act[:, None])[:, 0], 0.0)


# ---- play ---------------------------------------------------------------------------------------------


def play(choose, games: int, seed: int) -> dict:
    env = ml2048_b200.VecGame(games, output="torch", sync_free=True, rng_mode="philox", track_merged=False)
    env.reset(seed)
    env.enable_episode_log(games)
    log = env.episode_log()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    steps = 0
    while True:
        env.prepare()
        env.step(choose(env.observations()[0]))
        steps += 1
        if steps % 64 == 0 and bool((log["max_tile"] > 0).all()):
            break
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    score = log["score"].cpu().numpy().astype(np.float64)
    length = log["steps"].cpu().numpy().astype(np.float64)
    mt = log["max_tile"].cpu().numpy().astype(np.int64)
    return {"games": games, "mean_score": float(score.mean()), "mean_length": float(length.mean()),
            "reached": {str(1 << k): float((mt >= k).mean()) for k in (11, 12, 13, 14)},
            "batched_steps": steps, "wall_s": wall, "us_per_batched_step": wall / steps * 1e6,
            "us_per_move": wall / float(length.sum()) * 1e6}


# ---- the alternative mapping, in a child process -------------------------------------------------------


def child_main(path: str) -> None:
    d = torch.load(path)
    boards, weights = d["boards"].cuda(), d["weights"].cuda()
    res = {"depth1_us": time_depth1(boards, weights, d["sizes"], lambda m: max(2, (1 << 22) // m))}
    o = ops.ntuple_expectimax(boards, weights, STANDARD_4X6, depth=1, two_prob=TWO_PROB)
    torch.save({k: v.cpu() for k, v in o.items()}, path + ".out")
    print(json.dumps(res))


def alternative_mapping(tmp: str, boards, weights, sizes) -> dict:
    so = os.path.join(tmp, "libml2048_b200_warp_per_board.so")
    subprocess.run([nvcc_path(), *NVCC_FLAGS, "-DML2048_EXPECTIMAX_WARP_PER_BOARD", "-o", so, SRC, HOST_SRC, HOST_UNPACK_SRC,
                    COMPRESSIBLE_SRC], check=True)
    path = os.path.join(tmp, "alt_inputs.pt")
    torch.save({"boards": boards.cpu(), "weights": weights.cpu(), "sizes": sizes}, path)
    env = dict(os.environ, ML2048_LIB=so)
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path], env=env, capture_output=True, text=True, check=True)
    res = json.loads(out.stdout.strip().splitlines()[-1])
    theirs = torch.load(path + ".out")
    mine = ops.ntuple_expectimax(boards, weights, STANDARD_4X6, depth=1, two_prob=TWO_PROB)
    res["bit_identical"] = all(torch.equal(mine[k].cpu().view(torch.uint8), theirs[k].view(torch.uint8)) for k in mine)
    return res


def main() -> None:
    p = argparse.ArgumentParser()
    p.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    p.add_argument("--quick", action="store_true", help="small sizes and few games (a rehearsal, not a measurement)")
    p.add_argument("--child", default=None, help=argparse.SUPPRESS)
    args = p.parse_args()
    if args.child:
        child_main(args.child)
        return
    assert torch.cuda.is_available(), "needs a GPU"
    q = args.quick
    res = {"device": device_info(), "tuples": STANDARD_4X6, "two_prob": TWO_PROB, "reward": "normal"}
    t0 = time.perf_counter()
    net = NTupleNetwork()
    env = ml2048_b200.VecGame(1 << 14, output="torch", sync_free=True, rng_mode="philox")
    learner = TDAfterstateLearner(env, net)
    learner.reset(7)
    train_steps = 2000 if q else 100000
    for _ in range(train_steps):
        learner.step()
    torch.cuda.synchronize()
    res["training"] = {"games": 1 << 14, "steps": train_steps, "seconds": time.perf_counter() - t0}
    w = net.weights

    # steady-state boards of the network's own greedy play
    m_max = 1 << (16 if q else 20)
    genv = ml2048_b200.VecGame(m_max, output="torch", sync_free=True, rng_mode="philox")
    player = TDAfterstateLearner(genv, net, alpha=0.0)
    player.reset(3)
    for _ in range(200 if q else 1500):
        player.step()
    genv.prepare()
    boards = genv.observations()[0].clone()
    del player, genv
    res["boards"] = {"games": m_max, "greedy_steps": 200 if q else 1500,
                     "mean_empty_cells": float((boards == 0).sum(1).float().mean())}

    d1_sizes = [12, 14, 16] if q else [12, 14, 16, 18, 20]
    d2_sizes = [10, 12] if q else [10, 12, 14]
    with tempfile.TemporaryDirectory() as tmp:
        res["gather_ceiling"] = gather_ceiling(tmp)
        kern = {"depth1": {}, "depth2": {}, "greedy": {}}
        for lg in d1_sizes:
            m = 1 << lg
            b = boards[:m].contiguous()
            leaves = tree_counts(b, 1)
            o = outs(m)
            us = time_graph(lambda: ops.ntuple_expectimax(b, w, STANDARD_4X6, depth=1, two_prob=TWO_PROB, action_dtype=torch.uint8, out=o),
                            max(2, (1 << 22) // m))
            go = {k: v for k, v in outs(m).items() if k != "q"}
            gus = time_graph(lambda: ops.ntuple_greedy(b, w, STANDARD_4X6, action_dtype=torch.uint8, out=go), max(4, (1 << 26) // m))
            g_leaves = int(ops.valid_actions(b).sum())
            kern["depth1"][lg] = {"us": us, "ns_per_board": min(us) * 1e3 / m, "leaves_per_board": leaves / m,
                                  "lookups_per_board": leaves * LOOKUPS_PER_LEAF / m,
                                  "lookups_per_s": leaves * LOOKUPS_PER_LEAF / (min(us) * 1e-6)}
            kern["greedy"][lg] = {"us": gus, "ns_per_board": min(gus) * 1e3 / m, "lookups_per_board": g_leaves * LOOKUPS_PER_LEAF / m,
                                  "lookups_per_s": g_leaves * LOOKUPS_PER_LEAF / (min(gus) * 1e-6)}
            print(f"depth 1 M=2^{lg}: {min(us):.1f} us, {kern['depth1'][lg]['lookups_per_board']:.0f} lookups/board, "
                  f"{kern['depth1'][lg]['lookups_per_s'] / 1e9:.1f} G lookups/s; greedy {min(gus):.1f} us", flush=True)
        for lg in d2_sizes:
            m = 1 << lg
            b = boards[:m].contiguous()
            leaves = tree_counts(b, 2)
            o = outs(m)
            us = time_graph(lambda: ops.ntuple_expectimax(b, w, STANDARD_4X6, depth=2, two_prob=TWO_PROB, action_dtype=torch.uint8, out=o),
                            max(2, (1 << 16) // m))
            kern["depth2"][lg] = {"us": us, "ns_per_board": min(us) * 1e3 / m, "leaves_per_board": leaves / m,
                                  "lookups_per_board": leaves * LOOKUPS_PER_LEAF / m,
                                  "lookups_per_s": leaves * LOOKUPS_PER_LEAF / (min(us) * 1e-6)}
            print(f"depth 2 M=2^{lg}: {min(us):.1f} us, {kern['depth2'][lg]['lookups_per_board']:.0f} lookups/board, "
                  f"{kern['depth2'][lg]['lookups_per_s'] / 1e9:.1f} G lookups/s", flush=True)
        res["kernels"] = kern

        # the composed baseline
        m = 1 << 14
        b = boards[:m].contiguous()
        k_out = ops.ntuple_expectimax(b, w, STANDARD_4X6, depth=1, two_prob=TWO_PROB)
        c_act, c_val = composed_depth1(b, w)
        cus = time_eager(lambda: composed_depth1(b, w), 3)  # boolean indexing synchronises: not capturable
        res["composed_depth1"] = {"games": m, "us": cus, "kernel_us": kern["depth1"][14]["us"],
                                  "slower_than_kernel": min(cus) / min(kern["depth1"][14]["us"]),
                                  "action_mismatches": int((c_act != k_out["action"]).sum()),
                                  "value_bit_mismatches": int((c_val.view(torch.int32) != k_out["value"].view(torch.int32)).sum())}
        print("composed:", res["composed_depth1"], flush=True)

        res["alternative_warp_per_board"] = alternative_mapping(tmp, boards[:1 << d1_sizes[-1]].contiguous(), w, d1_sizes)
        print("alternative:", res["alternative_warp_per_board"], flush=True)

    # play strength
    n_games, n_games2 = (256, 64) if q else (4096, 1024)
    res["play"] = {
        "greedy": play(lambda x: net.greedy(x, action_dtype=torch.uint8)["action"], n_games, 11),
        "depth1": play(lambda x: net.expectimax(x, depth=1, action_dtype=torch.uint8)["action"], n_games, 11),
        "depth2": play(lambda x: net.expectimax(x, depth=2, action_dtype=torch.uint8)["action"], n_games2, 11),
        "greedy_same_games_as_depth2": play(lambda x: net.greedy(x, action_dtype=torch.uint8)["action"], n_games2, 11),
    }
    for k, v in res["play"].items():
        print(k, v, flush=True)

    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "expectimax_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    lines = [f"device: {res['device']}", f"training: {res['training']}", f"boards: {res['boards']}",
             f"gather ceilings: " + ", ".join(f"{k} {v['lookups_per_s'] / 1e9:.1f} G/s" for k, v in res["gather_ceiling"].items())]
    for depth in ("depth1", "depth2", "greedy"):
        for lg, r in kern[depth].items():
            lines.append(f"{depth} M=2^{lg}: {min(r['us']):.1f} us ({', '.join(f'{x:.1f}' for x in r['us'])}), {r['ns_per_board']:.1f} ns/board, "
                         f"{r.get('leaves_per_board', r['lookups_per_board'] / LOOKUPS_PER_LEAF):.1f} leaves/board, "
                         f"{r['lookups_per_board']:.0f} lookups/board, {r['lookups_per_s'] / 1e9:.1f} G lookups/s")
    lines.append(f"composed depth 1: {res['composed_depth1']}")
    lines.append(f"alternative mapping (warp per board): {res['alternative_warp_per_board']}")
    for k, v in res["play"].items():
        lines.append(f"play {k}: {v}")
    with open(os.path.join(args.out_dir, "expectimax_bench.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
