#!/usr/bin/env python
"""
bench.py -- env steps/sec of the VecGame hot path on N B200s (one JSON line, see the driver contract).

Workload (BASELINE.json configs[2]/[3]): M = 2^24 games per GPU, random-valid-action rollout,
one "step" = prepare() (auto-reset of finished games) + step() (move, reward/score, spawn, mask,
terminal flag) with the fp32 one-hot observation fused, replay (bit-exact) spawn tables, boards in
steady state after a 256-step burn-in.  Games are sharded over the ranks by global slot; the data
path has no collective, episode statistics are all-reduced once at the end (weak scaling).

  value      whole-job env-steps/s, device-timed (CUDA events), state resident in HBM
  e2e        same metric through the reference-facing API with HOST buffers: actions H2D from pinned
             memory, board/mask/reward/terminated D2H every step
  roofline   step kernel: algorithmic bytes (SURVEY.md section 8d: 59 + 1024 = 1083 B per env step) over its
             CUDA-event duration, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline / --impl reference
             the reference's own Numba VecGame (unmodified modules staged under oracle/_ref by oracle/make_ref.py,
             numba.set_num_threads(all host threads), BASELINE.md section 3 protocol) -- kind "reference"; the C/OpenMP
             port of the oracle is reported beside it ("cpu_port") and is the fallback when numba or the staged tree
             is missing (kind "port")
  shard_check (N > 1) before the timed region every rank plays its shard of a small global batch with globally
             slot-ordered ids (VecGame.shard()), rank 0 also plays the whole batch: boards, ids, scores, steps and the
             all-reduced statistics must be identical, otherwise the run fails
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
BYTES_CORE = 59          # SURVEY.md section 8(d): 25 B read + 34 B written per env step
BYTES_ONEHOT_F32 = 1024  # fp32 (16 classes x 16 cells) observation written per env step
BURN_IN = 256            # steps from reset() to steady-state boards (SURVEY.md section 8d, config 3)
STATS_EVERY = 64         # BASELINE configs[3]: the episode statistics are all-reduced every 64 steps (24 integers)
DUMP_GAMES = 1 << 15     # --dump-outputs: games sampled from the batch (1 KiB of fp32 one-hot + 0.2 KiB of other fields each)
DUMP_SEED = 2048         # --dump-outputs: seed of that sample, so that the same --games-per-gpu always gives the same slots


def parse_args() -> argparse.Namespace:
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=100)
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--impl", choices=["b200", "reference"], default="b200")
    p.add_argument("--games-per-gpu", type=int, default=1 << 24)
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--no-extras", action="store_true", help="skip the secondary measurements (core-only, small M)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-shard-check", action="store_true", help="profiling runs: skip the pre-timing shard self-check")
    p.add_argument("--no-fused-reset", action="store_true",
                   help="timed region: prepare() and step_random() as two calls instead of step_random(auto_reset=True)")
    p.add_argument("--cpu-games", type=int, default=0,
                   help="games per CPU step of the reference arm (0 = the GPU arm's games per GPU, halved until the run fits --ref-budget-s)")
    p.add_argument("--ref-budget-s", type=float, default=420.0, help="wall-clock budget of the --impl reference run")
    p.add_argument("--ref-kind", choices=["auto", "reference", "port"], default="auto",
                   help="CPU arm: the staged Numba reference (oracle/_ref), the C port (oracle/), or the first that is available")
    p.add_argument("--burn-in", type=int, default=BURN_IN, help="untimed steps from reset() to steady state")
    p.add_argument("--clock-interval-ms", type=float, default=50.0, help="NVML sampling period during the timed region")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed step returned (a fixed sample of the games) as "
                        "DIR/<name>.npy in float32 or float64, to compare two builds output for output; rank 0 only")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def workload_name(games_per_gpu: int, burn_in: int = BURN_IN) -> str:
    return (f"random-valid-action rollout, M={games_per_gpu} games/GPU (2^{games_per_gpu.bit_length() - 1}), "
            "prepare(auto-reset)+step+spawn+mask+terminal fused with fp32 one-hot obs, replay (bit-exact) tables, "
            f"steady state after {burn_in}-step burn-in")


# -------------------------------------------------------------------------------------------------
# CPU baseline (oracle port) -- also the --impl reference arm
# -------------------------------------------------------------------------------------------------


def time_cpu_port(games: int, steps: int, warmup: int, seed: int, budget_s: float | None = None) -> dict:
    """prepare()+step() of the CPU port on all host threads; actions (the policy) are generated outside
    the timed spans (BASELINE.md section 3 protocol).  Returns steps/s and what was run."""
    from oracle import oracle as orc

    lib = orc.load_lib()
    # all host threads this process may use (torchrun exports OMP_NUM_THREADS=1: override it for the CPU arm)
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    lib.orc_set_num_threads(avail)
    cores = int(lib.orc_num_threads())
    env = orc.OracleVecGame(games, "normal")
    env.reset(seed)
    import numpy as np

    acts = np.empty((games,), dtype=np.int64)
    # a short burn-in so that resets occur; the full 256-step burn-in would dominate the CPU budget
    for t in range(warmup):
        env.prepare()
        env.random_valid_actions(1000 + t, acts)
        env.step(acts)
    spent = 0.0
    done = 0
    t_start = time.perf_counter()
    for t in range(steps):
        t0 = time.perf_counter()
        env.prepare()
        t1 = time.perf_counter()
        env.random_valid_actions(t, acts)  # policy: untimed
        t2 = time.perf_counter()
        env.step(acts)
        t3 = time.perf_counter()
        spent += (t1 - t0) + (t3 - t2)
        done += 1
        if budget_s is not None and time.perf_counter() - t_start > budget_s:
            break
    return {
        "value": games * done / spent,
        "ms_per_step": 1e3 * spent / done,
        "steps": done,
        "cores": cores,
        "games": games,
        "sample": f"CPU port of the reference (oracle/vecgame_oracle.c, OpenMP, {cores} threads): prepare()+step() on "
                  f"M={games} games x {done} steps after {warmup} warm-up steps from reset(seed={seed}), random-valid "
                  "actions generated outside the timed spans",
    }


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def numba_reference_available() -> str | None:
    """None when the staged reference can be timed here, else the reason it cannot."""
    try:
        from oracle import make_ref

        if not make_ref.available():
            return "oracle/_ref is not staged (python -m oracle.make_ref, run by __graft_entry__.build())"
        import numba  # noqa: F401
    except Exception as exc:  # noqa: BLE001
        return f"{type(exc).__name__}: {exc}"
    return None


def time_numba_reference(games: int, steps: int, warmup: int, seed: int, budget_s: float | None = None,
                         threads: int | None = None) -> dict:
    """The reference's own ``VecGame`` (game_numba.py, unmodified, imported from oracle/_ref) timed per BASELINE.md
    section 3: ``numba.set_num_threads(all host threads)``, one untimed JIT pass, then ``prepare()`` -> random valid actions
    (generated OUTSIDE the timed spans, semantics of policy/random.py:24) -> ``step(actions)``, ``time.perf_counter``
    around prepare()+step().  When ``budget_s`` is given the batch is halved until the projected run (first prepare() of
    all M games in interpreted Python + warm-up + timed steps) fits it."""
    os.environ.pop("OMP_NUM_THREADS", None)  # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses all host threads
    import numba
    import numpy as np

    from oracle import make_ref
    from oracle import oracle as orc

    gn = make_ref.import_reference()
    cores = threads or host_threads()
    cores = min(cores, numba.config.NUMBA_NUM_THREADS)
    numba.set_num_threads(cores)
    lib = orc.load_lib()  # only the untimed random-valid policy below comes from oracle/
    lib.orc_set_num_threads(cores)

    # JIT pass + cost probe on a small instance (compiled functions are cached per signature, the big instance reuses them)
    probe_m = 1 << 14
    vg = gn.VecGame(probe_m)
    vg.reset(seed)
    acts = np.zeros((probe_m,), np.int64)
    vg.prepare()
    vg.step(acts)
    vg.reset(seed)
    t0 = time.perf_counter()
    vg.prepare()  # all probe_m games created: the interpreted per-slot loop of game_numba.py:634-656
    per_reset = (time.perf_counter() - t0) / probe_m
    lib.orc_random_valid_actions(vg._data.ctypes.data, probe_m, 1, acts.ctypes.data)
    t0 = time.perf_counter()
    vg.step(acts)
    per_game_step = max((time.perf_counter() - t0) / probe_m, 2e-9)
    del vg

    asked = games
    if budget_s is not None:
        def projected(m):  # large batches go DRAM-bound: allow 4x the probe's per-game step cost
            return m * (per_reset + (warmup + steps) * (4 * per_game_step + 0.0093 * per_reset))

        while games > (1 << 16) and projected(games) > budget_s:
            games //= 2

    vg = gn.VecGame(games)
    vg.reset(seed)
    acts = np.empty((games,), np.int64)
    t0 = time.perf_counter()
    for t in range(warmup):
        vg.prepare()
        lib.orc_random_valid_actions(vg._data.ctypes.data, games, 1000 + t, acts.ctypes.data)
        vg.step(acts)
    warm_s = time.perf_counter() - t0
    spent = step_only = 0.0
    done = 0
    for t in range(steps):
        t0 = time.perf_counter()
        vg.prepare()
        t1 = time.perf_counter()
        lib.orc_random_valid_actions(vg._data.ctypes.data, games, t, acts.ctypes.data)  # policy: untimed
        t2 = time.perf_counter()
        vg.step(acts)
        t3 = time.perf_counter()
        spent += (t1 - t0) + (t3 - t2)
        step_only += t3 - t2
        done += 1
    cpu_model = ""
    try:
        with open("/proc/cpuinfo") as fh:
            cpu_model = next((ln.split(":", 1)[1].strip() for ln in fh if ln.startswith("model name")), "")
    except OSError:
        pass
    shrunk = "" if games == asked else f" (asked for M={asked}; halved to fit the {budget_s:.0f} s budget)"
    return {
        "value": games * done / spent,
        "step_only_value": games * done / step_only,
        "ms_per_step": 1e3 * spent / done,
        "steps": done,
        "cores": cores,
        "games": games,
        "kind": "reference",
        "numba": numba.__version__,
        "threading_layer": numba.threading_layer(),
        "cpu_model": cpu_model,
        "warmup_s": warm_s,
        "sample": f"reference Numba VecGame (game_numba.py unmodified, staged in oracle/_ref; numba {numba.__version__}, "
                  f"{numba.threading_layer()} layer, {cores} of {os.cpu_count()} host threads, {cpu_model}): prepare()+step() on "
                  f"M={games} games x {done} steps{shrunk} after the all-games first prepare() and {warmup} warm-up steps "
                  f"from reset(seed={seed}), default reward_fn_normal, random-valid actions generated outside the timed spans",
    }


def make_config(args: argparse.Namespace, world: int) -> dict:
    """What the workload is -- a function of the command line only, so that both arms print the SAME config."""
    m = args.games_per_gpu
    return {
        "workload": workload_name(m, args.burn_in),
        "games_per_gpu": m,
        "global_games": m * world,
        "sharding": f"dp{world}: contiguous global slots, no data-path collective; episode statistics (24 integers: max-tile "
                    f"histogram, episodes, score/step sums, max score) all-reduced every min({STATS_EVERY}, steps) steps inside the "
                    "timed region",
        "l2": "inputs larger than L2 (boards 268 MB, one-hot 17 GB per GPU)",
        "rng": "replay tables (bit-exact mode); actions: uniform over valid, Philox, in-kernel",
    }


def time_cpu_arm(kind: str, games: int, steps: int, warmup: int, seed: int, budget_s: float | None) -> dict:
    """kind: "reference" (staged Numba VecGame), "port" (C/OpenMP oracle) or "auto" (the reference when it can run here)."""
    why_not = numba_reference_available() if kind in ("auto", "reference") else "port requested"
    if kind == "reference" and why_not:
        raise RuntimeError(f"--ref-kind reference: {why_not}")
    if why_not is None:
        return time_numba_reference(games, steps, warmup, seed, budget_s=budget_s)
    res = time_cpu_port(games, steps, warmup, seed)
    res["kind"] = "port"
    res["sample"] += f" [Numba reference unavailable: {why_not}]" if kind == "auto" else ""
    return res


def run_reference_arm(args: argparse.Namespace) -> None:
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return  # under torchrun only rank 0 runs the CPU arm
    warm = max(args.warmup, 3)
    games = args.cpu_games or args.games_per_gpu
    res = time_cpu_arm(args.ref_kind, games, args.steps, warm, args.seed, args.ref_budget_s)
    baseline = {k: res[k] for k in ("value", "cores", "kind", "sample") if k in res}
    baseline["unit"] = UNIT
    for k in ("step_only_value", "numba", "threading_layer", "cpu_model", "games"):
        if k in res:
            baseline[k] = res[k]
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": res["value"],
        "unit": UNIT,
        "n_gpus": args.gpus,
        "steps": res["steps"],
        "warmup": warm,
        "ms_per_step": res["ms_per_step"],
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "u8",
        "data": "synthetic",
        "config": make_config(args, max(world, args.gpus)),
        "cpu_baseline": baseline,
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if res.get("kind") == "reference":
        # second line of evidence: the C/OpenMP port of the oracle on the same batch (bounded to ~10 s)
        try:
            port = time_cpu_port(min(res["games"], 1 << 22), 40, 3, args.seed, budget_s=10.0)
            line["cpu_port"] = {"value": port["value"], "unit": UNIT, "cores": port["cores"], "kind": "port", "sample": port["sample"]}
        except Exception as exc:  # noqa: BLE001
            line["cpu_port"] = {"unavailable": repr(exc)}
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------------
# clocks
# -------------------------------------------------------------------------------------------------


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU periodically through NVML while running."""

    REASONS = {
        0x8: "hw_slowdown",
        0x40: "hw_thermal_slowdown",
        0x20: "sw_thermal_slowdown",
        0x4: "sw_power_cap",
        0x80: "hw_power_brake_slowdown",
    }

    def __init__(self, index: int, interval_s: float = 0.05):
        super().__init__(daemon=True)
        self.index = index
        self.interval_s = interval_s
        self.samples: list[int] = []
        self.reasons: set[str] = set()
        self.max_mhz = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = None
            try:
                import torch

                pr = torch.cuda.get_device_properties(index)
                bus = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
                self._h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self) -> None:
        if not self.ok:
            return
        nv = self._nv
        while not self._halt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                bits = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
                for bit, name in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.interval_s)

    def stop(self) -> dict:
        self._halt.set()
        if self.is_alive():
            self.join(timeout=2)
        med = sorted(self.samples)[len(self.samples) // 2] if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# -------------------------------------------------------------------------------------------------
# the B200 arm
# -------------------------------------------------------------------------------------------------


def load_peaks() -> tuple[float, str]:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_ncu_traffic(games: int):
    """dram bytes per launch of the fused step kernel from the committed ncu summary, if it matches M."""
    path = os.path.join(ROOT, "profiles", "step_kernel_traffic.json")
    try:
        with open(path) as fh:
            d = json.load(fh)
        per_game = d.get("dram_bytes_per_game_fused_f32")
        return None if per_game is None else float(per_game) * games
    except Exception:
        return None


def shard_check(ml2048_b200, torch, dist, dev, rank: int, world: int, seed: int) -> dict:
    """Pre-timing self-check of the sharded path.  A small global batch is played (a) sharded: every rank owns the
    contiguous global slots [rank*s, (rank+1)*s) and calls ``VecGame.shard()``, so that prepare() exchanges the per-rank
    reset counts (one all_gather) and game ids are globally slot-ordered like in one reference process
    (game_numba.py:641-644); (b) whole, on rank 0.  The in-kernel policy's Philox stream and the replay tables are keyed
    by the GLOBAL slot, so both runs must agree bit for bit: boards, masks, ids, scores, steps -- compared on rank 0 after an
    all_gather of the shards -- and the all-reduced episode statistics (RunnerStats.combine, runner.py:181-189) must
    equal the whole run's.  With one rank the same comparison runs in-process over two shards (ids per shard)."""
    from ml2048_b200.sharding import reduce_episode_stats

    s, steps = 40000, 180
    total = s * max(world, 2)
    fields = ("board", "valid", "id", "score", "step", "terminated")

    def play(env):
        env.reset(seed + 11)
        for _ in range(steps):
            env.prepare()
            env.step_random()
        cur = env._cur
        return {"board": env._board[cur].clone(), "valid": env._valid[cur].clone(), "id": env._id.clone(),
                "score": env._score.contiguous().view(torch.int32).clone(), "step": env._step.contiguous().clone(),
                "terminated": env._terminated.clone()}

    def make(size, base):
        return ml2048_b200.VecGame(size, ml2048_b200.reward_fn_improved, output="torch", slot_base=base, sync_free=True, device=dev)

    out = {"games": total, "steps": steps, "fields": list(fields) + ["episode_stats"]}
    if world == 1:
        whole_env = make(total, 0)
        whole = play(whole_env)
        parts, stats = [], torch.zeros((24,), dtype=torch.int64, device=dev)
        for r in range(2):
            e = make(s, r * s)
            parts.append(play(e))
            t = e.episode_stats_tensor()
            stats[:23] += t[:23]
            stats[23] = torch.maximum(stats[23], t[23])
        bad = [k for k in fields if k != "id" and not torch.equal(torch.cat([p[k] for p in parts]), whole[k])]
        if not torch.equal(stats, whole_env.episode_stats_tensor()):
            bad.append("episode_stats")
        out["mode"] = "1 rank: two in-process shards against the whole batch (ids are per shard and not compared)"
        out["episodes"] = int(stats[20].item())
    else:
        env = make(s, rank * s)
        env.shard()
        mine = play(env)
        stats = reduce_episode_stats(env.episode_stats_tensor())
        gathered = {}
        for k in fields:
            buf = torch.empty((world,) + tuple(mine[k].shape), dtype=mine[k].dtype, device=dev)
            dist.all_gather_into_tensor(buf, mine[k].contiguous())
            gathered[k] = buf.reshape((-1,) + tuple(mine[k].shape[1:]))
        bad = []
        if rank == 0:
            whole_env = make(total, 0)
            whole = play(whole_env)
            bad = [k for k in fields if not torch.equal(gathered[k], whole[k])]
            if not torch.equal(stats, whole_env.episode_stats_tensor()):
                bad.append("episode_stats")
            if env._game_count != whole_env._game_count:
                bad.append("game_count")
        flag = torch.tensor([len(bad)], dtype=torch.int64, device=dev)
        dist.broadcast(flag, src=0)
        if int(flag.item()) and rank != 0:
            bad = ["(see rank 0)"]
        out["mode"] = f"{world} NCCL ranks, VecGame.shard(): globally slot-ordered ids, shards all-gathered and compared on rank 0"
        out["episodes"] = int(stats[20].item())
    out["result"] = "ok" if not bad else "MISMATCH in " + ", ".join(bad)
    return out


def pcie_ceiling(torch, dist, dev, world: int, h2d_bytes: int, d2h_bytes: int, reps: int = 6) -> dict:
    """Bare pinned-memory copies of one e2e step's bytes (no kernels, no Python between them), all ranks at once: the
    ceiling the host-buffer path can reach on this box.  H2D and D2H run on two streams like the pipeline's."""
    host_in = torch.empty((max(h2d_bytes, 1),), dtype=torch.uint8, pin_memory=True)
    host_out = torch.empty((max(d2h_bytes, 1),), dtype=torch.uint8, pin_memory=True)
    dev_in = torch.empty_like(host_in, device=dev)
    dev_out = torch.zeros((max(d2h_bytes, 1),), dtype=torch.uint8, device=dev)
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    times = {"both": [], "d2h": [], "h2d": []}
    for which in ("both", "d2h", "h2d"):
        for _ in range(reps):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if which in ("both", "h2d"):
                with torch.cuda.stream(s_in):
                    dev_in.copy_(host_in, non_blocking=True)
            if which in ("both", "d2h"):
                with torch.cuda.stream(s_out):
                    host_out.copy_(dev_out, non_blocking=True)
            torch.cuda.synchronize()
            times[which].append(time.perf_counter() - t0)
    best = {k: min(v) for k, v in times.items()}
    if world > 1:
        t = torch.tensor([best["both"], best["d2h"], best["h2d"]], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        best = dict(zip(("both", "d2h", "h2d"), [float(x) for x in t.tolist()]))
    return {
        "ceiling_gbs": world * (h2d_bytes + d2h_bytes) / best["both"] / 1e9,
        "d2h_alone_gbs": world * d2h_bytes / best["d2h"] / 1e9,
        "h2d_alone_gbs": world * h2d_bytes / best["h2d"] / 1e9,
        "ms_per_step_at_ceiling": best["both"] * 1e3,
    }


def dump_outputs(env, result, out_dir: str, slot_base: int) -> None:
    """Write what the last timed step returned, so that two builds can be compared output for output on the same command
    line: the fields of its ``VecStepResult``, the fused one-hot observation and the game ids for a fixed, seeded sample of
    DUMP_GAMES games (their global slots in ``slot.npy``), which of those games the step's auto-reset restarted, how many
    it restarted in all, and the episode statistics of the whole batch.  Integers wider than 16 bits are written as
    float64 (exact), everything else as float32: at most ~40 MB."""
    import numpy as np
    import torch

    m = env._size
    sel = np.sort(np.random.default_rng(DUMP_SEED).choice(m, size=min(m, DUMP_GAMES), replace=False))
    idx = torch.from_numpy(sel).to(env.device)
    out = {"slot": torch.from_numpy(sel + slot_base)}
    for key in result.keys():
        try:
            out[key] = result[key][idx]
        except KeyError:  # `merged` is not tracked on the timed path
            continue
    out["onehot"] = env.observations_onehot()[idx]
    out["id"] = env._id[idx]
    (reset,) = env.last_reset()
    was_reset = torch.zeros((m,), dtype=torch.bool, device=env.device)
    was_reset[reset.long()] = True
    out["reset"] = was_reset[idx]
    out["reset_count"] = torch.tensor([reset.numel()])
    out["episode_stats"] = env.episode_stats_tensor()
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        t = t.cpu()
        wide = t.dtype == torch.float64 or (not t.dtype.is_floating_point and t.dtype.itemsize > 2)
        np.save(os.path.join(out_dir, f"{name}.npy"), t.to(torch.float64 if wide else torch.float32).numpy())


def run_b200_arm(args: argparse.Namespace) -> None:
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback in ml2048_b200)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else "single process: not bound"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import ml2048_b200
    from ml2048_b200.sharding import reduce_episode_stats
    from ml2048_b200.vecgame import stats_to_dict

    m = args.games_per_gpu
    k_steps, warm = args.steps, max(args.warmup, 3)
    slot_base = rank * m

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- sharded-path self-check (before anything is timed) ------------------------------------
    check = ({"result": "skipped (--no-shard-check)"} if args.no_shard_check
             else shard_check(ml2048_b200, torch, dist, dev, rank, world, args.seed))
    if check["result"] != "ok" and not args.no_shard_check:
        raise SystemExit(f"shard_check failed on rank {rank}: {check}")
    torch.cuda.empty_cache()

    # ---- device-resident arm: `value` --------------------------------------------------------
    env = ml2048_b200.VecGame(m, ml2048_b200.reward_fn_normal, output="torch", onehot="f32", track_merged=False,
                              slot_base=slot_base, sync_free=True, device=dev)
    env.reset(args.seed)
    for _ in range(args.burn_in):
        env.prepare()
        env.step_random()
    torch.cuda.synchronize()
    snapshot = None if args.no_e2e else env.state_dict()

    stats_every = min(STATS_EVERY, k_steps)
    pending = []

    def reduce_stats_async(e):
        """The job's only collective: SUM of the max-tile histogram + episode/score/step sums, MAX of the best score
        (RunnerStats.combine, runner.py:181-189), issued on NCCL's stream; the caller waits for it before the timed
        region closes."""
        snap = e.episode_stats_tensor()
        sums, mx = snap[:23].clone(), snap[23:].clone()
        if world > 1:
            pending.append((dist.all_reduce(sums, op=dist.ReduceOp.SUM, async_op=True),
                            dist.all_reduce(mx, op=dist.ReduceOp.MAX, async_op=True), sums, mx))
        else:
            pending.append((None, None, sums, mx))

    fused = not args.no_fused_reset
    last_result = [None]  # what the last step returned to its caller (--dump-outputs)

    def run_steps(e, n: int, kernel_events=None) -> int:
        reduces = 0
        for i in range(n):
            if not fused:
                e.prepare()
            if kernel_events is not None:
                kernel_events[i][0].record()
            # fused: the auto-reset rides inside the step kernel (same arrays afterwards as prepare() + step_random(),
            # tests/test_fused_autoreset.py); a one-block-per-32k-games scan of the terminated flags ranks the resets first
            last_result[0] = e.step_random(auto_reset=fused)
            if kernel_events is not None:
                kernel_events[i][1].record()
            if kernel_events is not None and (i + 1) % stats_every == 0:
                reduce_stats_async(e)
                reduces += 1
        for w0, w1, _, _ in pending:  # the reductions finish INSIDE the timed region
            if w0 is not None:
                w0.wait()
                w1.wait()
        return reduces

    run_steps(env, warm)
    # first use of a torch op / an NCCL communicator loads kernels and connects ranks (tens to hundreds of ms):
    # do both once before the timed region, which repeats them every `stats_every` steps
    reduce_stats_async(env)
    for w0, w1, _, _ in pending:
        if w0 is not None:
            w0.wait()
            w1.wait()
    pending.clear()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k_steps)]
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local_rank, args.clock_interval_ms * 1e-3)
    barrier()
    sampler.start()
    start.record()
    reduces_timed = run_steps(env, k_steps, kev)
    stop.record()
    barrier()
    clocks = sampler.stop()
    elapsed_ms = max_over_ranks(start.elapsed_time(stop))
    value = world * m * k_steps / (elapsed_ms * 1e-3)
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / k_steps
    kernel_ms = max_over_ranks(kernel_ms)
    gaps = sorted(kev[i][1].elapsed_time(kev[i + 1][0]) for i in range(k_steps - 1)) or [0.0]
    prepare_ms = gaps[len(gaps) // 2]  # median gap between step kernels = the auto-reset (a gap that holds a reduction is longer)
    timed_stats = torch.cat([pending[-1][2], pending[-1][3]]) if pending else None
    pending.clear()
    if os.environ.get("ML2048_BENCH_DEBUG"):
        print(f"[debug] prepare gaps ms: min {gaps[0]:.3f} p50 {gaps[len(gaps)//2]:.3f} p90 {gaps[int(len(gaps)*0.9)]:.3f} max {gaps[-1]:.3f}",
              file=sys.stderr)
    if args.dump_outputs and rank == 0:
        dump_outputs(env, last_result[0], args.dump_outputs, slot_base)

    # the collective by itself: the same two all-reduces, blocking, back to back (device-timed, max over ranks)
    collective_ms = None
    if world > 1:
        snap = env.episode_stats_tensor()
        sums, mx = snap[:23].clone(), snap[23:].clone()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        c0.record()
        for _ in range(10):
            dist.all_reduce(sums, op=dist.ReduceOp.SUM)
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        c1.record()
        torch.cuda.synchronize()
        collective_ms = max_over_ranks(c0.elapsed_time(c1) / 10)

    peak, peak_src = load_peaks()
    bytes_per_launch = (BYTES_CORE + BYTES_ONEHOT_F32) * m
    achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm",
        "kernel": "step_kernel<replay, onehot f32> (move+reward+spawn+mask+terminal+one-hot" + (
            "+auto-reset; kernel_ms includes the ~3 us scan of the terminated flags that precedes it)" if fused else ")"),
        "achieved": achieved,
        "peak": peak,
        "peak_source": peak_src,
        "unit": "GB/s",
        "frac": achieved / peak,
        "traffic": load_ncu_traffic(m),
        "traffic_source": "profiles/step_kernel_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per game of this kernel from "
                          "the committed `ncu --set full` capture, times M -- a cross-reference, not a counter read in this run",
        "bytes_per_env_step": BYTES_CORE + BYTES_ONEHOT_F32,
        "kernel_ms": kernel_ms,
        "kernel_share_of_step": kernel_ms / (elapsed_ms / k_steps),
        "prepare_ms": prepare_ms,
    }

    # final statistics (the same 24-integer reduction once more, after the timed region)
    stats = reduce_episode_stats(env.episode_stats_tensor())
    stats_d = stats_to_dict(stats)

    extras = {}
    if not args.no_extras and rank == 0:
        extras = measure_extras(ml2048_b200, torch, dev, args.seed)

    # ---- end-to-end arm: host buffers through the reference-facing API -----------------------
    e2e = None
    if not args.no_e2e:
        # record the (valid, random) actions of the next warm+k steps of this exact trajectory, then
        # rewind the environment and replay them from pinned HOST memory through step(actions)
        env.load_state_dict(snapshot)
        total = warm + k_steps
        host_actions = torch.empty((total, m), dtype=torch.uint8, pin_memory=True)
        for t in range(total):
            env.prepare()
            env.step_random(return_actions=True)
            host_actions[t].copy_(env._actions_out, non_blocking=True)
        torch.cuda.synchronize()
        env.load_state_dict(snapshot)
        env.configure(output="numpy", sync_free=False)
        consumed = 0

        result_bytes = [0]

        def e2e_step(t: int) -> int:
            (idx,) = env.prepare()                # D2H: reset count + indices
            keys = ("state", "valid_actions", "reward", "terminated")  # D2H: what a rollout consumer reads
            res = env.step(host_actions[t], fetch=keys)  # H2D: M action bytes
            # bytes that crossed PCIe towards the host: the environment reports what it copied (valid_actions + terminated travel
            # as ONE packed byte per game and are expanded on the host, inside this timed call); else the arrays themselves
            got = getattr(env, "last_step_d2h_bytes", None)
            if got is None:
                got = sum(res[key].nbytes for key in keys)
            result_bytes[0] = sum(res[key].nbytes for key in keys) + idx.nbytes + 8
            return got + idx.nbytes + 8

        for t in range(warm):
            e2e_step(t)
        barrier()
        t0 = time.perf_counter()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        d2h = 0
        for t in range(warm, total):
            d2h += e2e_step(t)
        ev1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        e2e_ms = max_over_ranks(max(ev0.elapsed_time(ev1), wall_ms))
        # the replayed host actions were recorded from this very trajectory, so every one of them must be a valid move
        invalid_last = int(env._invalid.sum().item())
        # second regime: the policy lives on the GPU, the host only reads reward + terminated (5 B per game)
        env.load_state_dict(snapshot)  # rewind again: the recorded actions belong to this trajectory
        del snapshot
        light_steps = min(total - 3, 20)
        for t in range(3):
            env.prepare()
            env.step(host_actions[t], fetch=("reward", "terminated"))
        barrier()
        t0 = time.perf_counter()
        for t in range(3, 3 + light_steps):
            env.prepare()
            res = env.step(host_actions[t], fetch=("reward", "terminated"))
        torch.cuda.synchronize()
        light_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / light_steps
        invalid_last = max(invalid_last, int(env._invalid.sum().item()))
        h2d_step, d2h_step = int(m * world), int(d2h / k_steps * world)
        e2e = {
            "value": world * m * k_steps / (e2e_ms * 1e-3),
            "unit": UNIT,
            "h2d_bytes_per_step": h2d_step,
            "d2h_bytes_per_step": d2h_step,
            "result_bytes_per_step": int(result_bytes[0] * world),
            "d2h_note": "d2h_bytes_per_step = bytes copied device->host per step (board 16 B, reward 4 B, valid_actions + terminated as one "
                        "packed byte per game, reset indices); result_bytes_per_step = the host arrays the caller receives (25 B per game), "
                        "rebuilt from the packed byte by host threads inside the timed step",
            "ms_per_step": e2e_ms / k_steps,
            "invalid_moves_in_last_step": invalid_last,
            "light": {"value": world * m / (light_ms * 1e-3), "ms_per_step": light_ms,
                      "d2h": "reward + terminated only (5 B per game); observations stay on the device"},
            "api": "VecGame.prepare() -> (indices,); VecGame.step(uint8 actions in pinned host memory) -> "
                   "state, valid_actions, reward, terminated as host arrays",
        }
        # the e2e path's own roofline: what the box's PCIe/host-memory path carries when nothing but the copies runs
        del env
        torch.cuda.empty_cache()
        ceil = pcie_ceiling(torch, dist, dev, world, h2d_step // world, d2h_step // world)
        e2e["pcie_gbs"] = (h2d_step + d2h_step) / (e2e_ms / k_steps * 1e-3) / 1e9
        e2e["pcie_ceiling_gbs"] = ceil["ceiling_gbs"]
        e2e["frac"] = e2e["pcie_gbs"] / ceil["ceiling_gbs"]
        e2e["pcie"] = dict(ceil, how="bare pinned-memory copies of one step's bytes per rank (H2D and D2H on two streams), all "
                                     f"{world} rank(s) at once, best of 6, wall clock between synchronisations, max over ranks")

    cpu_baseline = cpu_port = None
    if not args.no_cpu_baseline and rank == 0 and world == 1:
        # bounded samples (the reference arm, `--impl reference`, runs the full batch): ~20 s of CPU work in all
        try:
            res = time_cpu_arm(args.ref_kind, 1 << 20, 24, 3, args.seed, budget_s=25.0)
        except Exception as exc:  # noqa: BLE001
            res = time_cpu_port(1 << 22, 40, 3, args.seed, budget_s=10.0)
            res["kind"] = "port"
            res["sample"] += f" [Numba reference failed: {exc!r}]"
        cpu_baseline = {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": res["kind"], "sample": res["sample"]}
        if res["kind"] == "reference":
            cpu_baseline["step_only_value"] = res["step_only_value"]
            port = time_cpu_port(1 << 22, 40, 3, args.seed, budget_s=8.0)
            cpu_port = {"value": port["value"], "unit": UNIT, "cores": port["cores"], "kind": "port", "sample": port["sample"]}

    if rank == 0:
        split = os.environ.get("ML2048_PREPARE", "").startswith("s")
        line = {
            "metric": METRIC,
            "value": value,
            "unit": UNIT,
            "n_gpus": world,
            "steps": k_steps,
            "warmup": warm,
            "ms_per_step": elapsed_ms / k_steps,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": "u8",
            "data": "synthetic",
            "config": make_config(args, world),
            "host_affinity": numa,
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": (2 if fused else 4 if split else 2) * k_steps,
            "launches_per_step": ("autoreset_scan_kernel, step_kernel with the auto-reset fused in" if fused
                                  else "prepare_count, prepare_scan, prepare_apply, step_kernel" if split
                                  else "prepare_fused_kernel (one cooperative launch), step_kernel"),
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "cpu_port": cpu_port,
            "shard_check": check["result"],
            "shard_check_detail": check,
            "collective": {
                "what": "all_reduce SUM int64[23] (max-tile histogram, episodes, score sum, step sum) + all_reduce MAX int64[1] "
                        "(best score), NCCL, issued asynchronously and waited for before the timed region closes",
                "every_steps": stats_every,
                "reduces_timed": reduces_timed,
                "collective_ms": collective_ms,
                "episodes_in_timed_reduce": None if timed_stats is None else int(timed_stats[20].item()),
            },
            "episode_stats": {k: (v.tolist() if hasattr(v, "tolist") else v) for k, v in stats_d.items()},
            "extras": extras,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_extras(ml2048_b200, torch, dev, seed: int) -> dict:
    """Secondary lines (not the headline): core-only path, Philox mode, narrower one-hot types, and the
    training shapes of run_train3.py (BASELINE configs[1]) replayed as a 16-step CUDA graph."""
    out = {}

    def timed(env, n, graph_steps=0, fused=False):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if graph_steps:
            roll = ml2048_b200.GraphedRollout(env, graph_steps, window=graph_steps * 16, auto_reset=fused)
            roll.replay(1)
            torch.cuda.synchronize()
            a.record()
            roll.replay(n // graph_steps)
            b.record()
        else:
            def one():
                if not fused:
                    env.prepare()
                env.step_random(auto_reset=fused)

            for _ in range(5):
                one()
            torch.cuda.synchronize()
            a.record()
            for _ in range(n):
                one()
            b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    for name, kw, m, n, graph_steps, fused in (
        ("core_only_replay_M2^24", dict(rng_mode="replay"), 1 << 24, 48, 0, True),
        ("core_only_replay_M2^24_separate_prepare", dict(rng_mode="replay"), 1 << 24, 48, 0, False),
        ("core_only_philox_M2^24", dict(rng_mode="philox"), 1 << 24, 48, 0, True),
        ("fused_bf16_onehot_M2^24", dict(rng_mode="replay", onehot="bf16"), 1 << 24, 48, 0, True),
        ("fused_u8_onehot_M2^24", dict(rng_mode="replay", onehot="u8"), 1 << 24, 48, 0, True),
        ("train_shape_M2048_fused_f32_eager", dict(rng_mode="replay", onehot="f32"), 2048, 192, 0, False),
        ("train_shape_M2048_fused_f32_graph16", dict(rng_mode="replay", onehot="f32"), 2048, 192, 16, False),
        ("train_shape_M2048_fused_f32_graph16_fused_reset", dict(rng_mode="replay", onehot="f32"), 2048, 192, 16, True),
        ("train_shape_M4096_fused_f32_graph16", dict(rng_mode="replay", onehot="f32"), 4096, 192, 16, False),
    ):
        env = ml2048_b200.VecGame(m, ml2048_b200.reward_fn_improved if m < 100000 else None, output="torch",
                                  track_merged=False, sync_free=True, device=dev, **kw)
        env.reset(seed)
        for _ in range(64 if m > 100000 else 128):
            env.prepare()
            env.step_random()
        ms = timed(env, n, graph_steps, fused)
        out[name] = {"us_per_step": ms * 1e3, "env_steps_per_s": m / (ms * 1e-3), "auto_reset": "fused into the step kernel" if fused
                     else "separate prepare() launch"}
        if m >= 1 << 24:
            out[name]["hbm_frac_whole_step_core_bytes"] = BYTES_CORE * m / (ms * 1e-3) / 1e9 / load_peaks()[0] if "onehot" not in kw else None
        if name == "core_only_replay_M2^24_separate_prepare":
            # the environment alone: actions GIVEN (recorded from this trajectory, device-resident), step kernel timed by itself
            snap = env.state_dict()
            k = 24
            acts = torch.empty((k, m), dtype=torch.uint8, device=dev)
            for t in range(k):
                env.prepare()
                env.step_random(return_actions=True)
                acts[t].copy_(env.sampled_actions)
            env.load_state_dict(snap)
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
            for t in range(k):
                env.prepare()
                ev[t][0].record()
                env.step(acts[t])
                ev[t][1].record()
            torch.cuda.synchronize()
            kms = sum(a.elapsed_time(b) for a, b in ev[4:]) / (k - 4)
            out["core_only_given_actions_step_kernel_M2^24"] = {
                "us_per_launch": kms * 1e3, "env_steps_per_s": m / (kms * 1e-3),
                "hbm_frac": BYTES_CORE * m / (kms * 1e-3) / 1e9 / load_peaks()[0]}
            del snap, acts
        del env
        torch.cuda.empty_cache()
    return out


def bind_to_gpu_numa_node(local_rank: int) -> str:
    """Pin this process to the CPUs NVML reports as local to its GPU, so that the pinned host buffers of the e2e arm are
    allocated (first touch) on the NUMA node the GPU's PCIe root hangs off.  Harmless when it cannot be done."""
    try:
        import pynvml
        import torch

        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(local_rank)
        bus = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cpus local to GPU {local_rank}"
    except Exception as exc:  # noqa: BLE001
        return f"not bound ({type(exc).__name__})"
    return "not bound"


def main() -> None:
    # the benchmark writes nothing into the tree it runs from (which may be read-only): not even bytecode of the modules
    # build() never imported, such as oracle/oracle.py of the CPU baseline
    sys.dont_write_bytecode = True
    args = parse_args()
    # exactly ONE line may reach stdout (the driver parses it): everything libraries print to fd 1 (NCCL's version
    # banner, for one) is sent to stderr, and the JSON line is written to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
