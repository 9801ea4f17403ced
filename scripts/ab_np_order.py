#!/usr/bin/env python
"""A/B of the nearest-plane update order (np_block, DESIGN.md 4.3) on the C2 step: runs
`python bench.py --workload c2 --no-extra --no-cpu-baseline` as subprocesses, alternating QF_NP_ORDER=right (the
right-looking order) and the default (left-looking inside each 4096-block), and writes the `value`, `e2e` and
`ms_per_step` samples of both arms with their medians, the card name and its power limit.
Usage: python scripts/ab_np_order.py [--rounds 3] [--out profiles/ab_np_order.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(order):
    env = dict(os.environ)
    env.pop("QF_NP_ORDER", None)
    if order == "right":
        env["QF_NP_ORDER"] = "right"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--no-extra", "--no-cpu-baseline"],
                         cwd=ROOT, env=env, check=True, capture_output=True, text=True).stdout
    line = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
    return {"value": line["value"], "e2e": line["e2e"]["value"], "ms_per_step": line["ms_per_step"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ab_np_order.json"))
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    arms = {"right": [], "left": []}
    for r in range(args.rounds):
        for order in ("right", "left"):
            s = run_bench(order)
            arms[order].append(s)
            print(f"round {r} {order}: {s}", flush=True)
    res = {"workload": "c2", "command": "python bench.py --workload c2 --no-extra --no-cpu-baseline", "card": card,
           "arms": {}}
    for order, samples in arms.items():
        res["arms"][order] = {
            "env": "QF_NP_ORDER=right" if order == "right" else "(default)",
            "samples": samples,
            "median": {k: statistics.median(s[k] for s in samples) for k in samples[0]},
            "spread": {k: max(s[k] for s in samples) - min(s[k] for s in samples) for k in samples[0]},
        }
    res["gain_value"] = res["arms"]["left"]["median"]["value"] / res["arms"]["right"]["median"]["value"] - 1
    res["gain_e2e"] = res["arms"]["left"]["median"]["e2e"] / res["arms"]["right"]["median"]["e2e"] - 1
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "gain_value", "gain_e2e")}), flush=True)


if __name__ == "__main__":
    main()
