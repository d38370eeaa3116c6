"""Same-box A/B of built trees on the flagship workload: bench.py run in each tree in turn, alternating, for N rounds.

    python scripts/gpu_l2_policy_ab.py --out DIR [--rounds 3] TREE_A TREE_B [TREE_C ...]

Each tree must already be built (python -m manual_whisper_b200.build).  A round runs, in every tree,
    bench.py --no-cpu-baseline --skip-e2e                      (8 batches in flight: value and roofline.in_step)
    bench.py --no-cpu-baseline --skip-e2e --streams 1 --no-extras   (the lone-batch step)
with --dump-outputs, so the token ids of every run can be compared byte for byte.  Prints, per tree, the median and
spread (min..max) of value, in_step.{ms_per_batch_step, cross_attention.ms, projection_gemms.ms} and the lone-batch
ms per decode step, whether every run's ids equal those of the first tree, the card's name and its power limit.
The JSON lines and ids go under --out; nothing is written inside the trees.  Runs are appended to --out/runs.jsonl and the
summary covers every run recorded there, so a comparison can be spread over several invocations.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

MODES = {"n8": ["--no-cpu-baseline", "--skip-e2e"],
         "solo": ["--no-cpu-baseline", "--skip-e2e", "--streams", "1", "--no-extras"]}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def run_bench(tree, mode, dump_dir):
    cmd = [sys.executable, "bench.py", "--gpus", "1", *MODES[mode], "--dump-outputs", dump_dir]
    t0 = time.time()
    r = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{tree} {mode}: exit {r.returncode}\n{r.stderr[-3000:]}")
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    res = json.loads(line)
    res["_wall_s"] = time.time() - t0
    return res


def metrics(res, mode):
    if mode == "solo":
        return {"solo_ms_per_step": res["ms_per_step"], "solo_value": res["value"]}
    st = res["roofline"]["in_step"]
    return {"value": res["value"], "ms_per_batch_step": st["ms_per_batch_step"],
            "cross_attention_ms": st["cross_attention"]["ms"], "projection_gemms_ms": st["projection_gemms"]["ms"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("trees", nargs="+")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import numpy as np
    trees = [os.path.abspath(t) for t in a.trees]
    names = [os.path.basename(t.rstrip("/")) or t for t in trees]
    assert len(set(names)) == len(names), "trees need distinct directory names"
    a.out = os.path.abspath(a.out)                      # bench.py runs inside each tree
    os.makedirs(a.out, exist_ok=True)
    print(f"card: {card()}", flush=True)
    same = {n: True for n in names}
    ref_ids, ids_of = {}, {}
    with open(os.path.join(a.out, "runs.jsonl"), "a") as log:
        for rnd in range(a.rounds):
            for mode in MODES:
                order = list(zip(trees, names))
                if rnd % 2:
                    order.reverse()                     # alternate which tree runs first
                for tree, name in order:
                    dump = os.path.join(a.out, f"ids_{name}_{mode}_{rnd}")
                    res = run_bench(tree, mode, dump)
                    ids = np.load(os.path.join(dump, "token_ids.npy"))
                    if mode not in ref_ids and name == names[0]:
                        ref_ids[mode] = ids
                    m = metrics(res, mode)
                    log.write(json.dumps({"tree": name, "mode": mode, "round": rnd, "card": card(), **m, "line": res}) + "\n")
                    log.flush()
                    print(f"round {rnd} {mode:4s} {name:12s} " + " ".join(f"{k}={v:.4g}" for k, v in m.items())
                          + f" ({res['_wall_s']:.0f} s)", flush=True)
                    ids_of[name, mode, rnd] = ids
            # ids of every tree against the first tree's, this round and mode
            for mode in MODES:
                for name in names:
                    ids = ids_of[name, mode, rnd]
                    if not (ids.shape == ref_ids[mode].shape and np.array_equal(ids, ref_ids[mode])):
                        same[name] = False
    print(f"\ncard: {card()}")
    got = {n: {} for n in names}
    with open(os.path.join(a.out, "runs.jsonl")) as f:
        for rec in map(json.loads, f):
            if rec["tree"] in got:
                for k, v in rec.items():
                    if k not in ("tree", "mode", "round", "card", "line"):
                        got[rec["tree"]].setdefault(k, []).append(v)
    summary = {}
    for name in names:
        row = {}
        for k, v in got[name].items():
            row[k] = {"median": statistics.median(v), "min": min(v), "max": max(v), "n": len(v)}
        row["ids_equal_first_tree"] = same[name]
        summary[name] = row
        print(f"{name}: ids equal to {names[0]}'s: {same[name]}")
        for k, s in row.items():
            if isinstance(s, dict):
                print(f"  {k:22s} median {s['median']:.4g}  spread {s['min']:.4g} .. {s['max']:.4g}  (n={s['n']})")
    with open(os.path.join(a.out, "summary.json"), "w") as f:
        json.dump({"card": card(), "trees": names, "summary": summary}, f, indent=1)


if __name__ == "__main__":
    main()
