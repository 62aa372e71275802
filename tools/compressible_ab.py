"""A/B of the one-hot observation in compressible against plain device memory, through bench.py itself.

Runs `bench.py --no-cpu-baseline --no-e2e` alternately with ML2048_ONEHOT_COMPRESSIBLE unset (compressible, the default)
and =0 (plain torch memory), --runs times each, every run dumping its outputs (--dump-outputs) to a directory of its own.
Every dumped array must be equal across all runs of both arms (same seed, same values); the tool prints the card's
name and power limit, each run's JSON line, and the median and min-max of `value` per arm, and writes it all as JSON.

    python tools/compressible_ab.py --runs 3 --out /tmp/compressible_ab [-- extra bench.py arguments]
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARMS = {"compressible": None, "plain": "0"}


def run_bench(arm: str, dump: str, extra: list[str]) -> dict:
    env = dict(os.environ)
    env.pop("ML2048_ONEHOT_COMPRESSIBLE", None)
    if ARMS[arm] is not None:
        env["ML2048_ONEHOT_COMPRESSIBLE"] = ARMS[arm]
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--no-cpu-baseline", "--no-e2e", "--dump-outputs", dump, *extra]
    out = subprocess.run(cmd, check=True, capture_output=True, text=True, env=env, cwd=ROOT).stdout
    return json.loads([line for line in out.splitlines() if line.startswith("{")][-1])


def main() -> None:
    p = argparse.ArgumentParser()
    p.add_argument("--runs", type=int, default=3, help="runs per arm (alternating)")
    p.add_argument("--out", default=None, help="directory for ab.json (default: print only)")
    p.add_argument("extra", nargs="*", help="more bench.py arguments (after --)")
    a = p.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print(f"card: {card}", flush=True)
    dumps = tempfile.mkdtemp(prefix="compressible_ab_")
    runs = []
    for r in range(a.runs):
        for arm in ARMS:
            d = os.path.join(dumps, f"{arm}_{r}")
            line = run_bench(arm, d, a.extra)
            runs.append({"arm": arm, "run": r, "dir": d, "value": line["value"], "line": line})
            print(json.dumps({"arm": arm, "run": r, "value": line["value"]}), flush=True)
    ref = runs[0]["dir"]
    names = sorted(f for f in os.listdir(ref) if f.endswith(".npy"))
    assert names, "bench.py dumped nothing"
    for run in runs[1:]:
        got = sorted(f for f in os.listdir(run["dir"]) if f.endswith(".npy"))
        assert got == names, (run["arm"], run["run"], got)
        for n in names:
            assert np.array_equal(np.load(os.path.join(ref, n)), np.load(os.path.join(run["dir"], n)), equal_nan=True), \
                f"{n} differs: {run['arm']} run {run['run']} against {runs[0]['arm']} run 0"
    print(f"outputs: all {len(names)} dumped arrays equal across {len(runs)} runs", flush=True)
    summary = {"card": card, "bench_args": ["--no-cpu-baseline", "--no-e2e", *a.extra], "outputs_equal": True, "arms": {}}
    for arm in ARMS:
        v = [r["value"] for r in runs if r["arm"] == arm]
        summary["arms"][arm] = {"median": statistics.median(v), "min": min(v), "max": max(v), "values": v}
        print(f"{arm:>12}: median {statistics.median(v) / 1e9:.3f} G env-steps/s (min {min(v) / 1e9:.3f}, max {max(v) / 1e9:.3f})")
    c, pl = summary["arms"]["compressible"], summary["arms"]["plain"]
    summary["median_ratio"] = c["median"] / pl["median"]
    summary["ranges_overlap"] = c["min"] <= pl["max"] and pl["min"] <= c["max"]
    print(f"compressible / plain median {summary['median_ratio']:.3f}, ranges overlap: {summary['ranges_overlap']}")
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        summary["runs"] = [{k: r[k] for k in ("arm", "run", "value", "line")} for r in runs]
        with open(os.path.join(a.out, "ab.json"), "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
