#!/usr/bin/env python3
"""Latency of unsampled pairs with per-base data (constraints, stacking pseudo-energies), to compare two commits.

    python tools/perbase_latency.py [--root DIR] [--reps 30] [--warmup 5] [--out FILE]

--root: the checkout whose ractip_b200 (and its built library) is loaded, default this one; run the tool once with
each of two checkouts, alternating, to compare them.  For MicA x ompA and OxyS x fhlA, four device batches of that
one pair, each created once and run with rp_batch_run + rp_batch_sync, alternated rep by rep, median of --reps after
--warmup:
  plain        no per-base data (band kernels)
  constrained  `x` on s1 1..5 and s2 1..5: all three problems on the general kernel's per-base instances
  shaped       seeded random reactivities (15 % missing) through rp_shape_deigan on both sequences: the same
  both         the two together
None is sampled.  Two clocks: the host clock around run + sync, and the library's CUDA events around the launches
(rp_timing::ms_total).  The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON
object (and writes it to --out).  Needs a GPU: there is no CPU fallback.
"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

HERE = Path(__file__).resolve().parent.parent


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=str(HERE))
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    root = Path(args.root).resolve()
    sys.path.insert(0, str(root))
    import numpy as np
    from ractip_b200 import ProbabilityStage, default_opts, shape_deigan

    seqs = json.loads((HERE / "tests" / "golden" / "bundled_pairs.json").read_text())["sequences"]
    rng = np.random.default_rng(7)

    def reactivities(n):
        r = rng.gamma(0.6, 0.8, size=n)
        r[rng.random(n) < 0.15] = -999.0
        return r

    stage = ProbabilityStage()
    o = default_opts()
    out = {"root": str(root), "card": card(), "reps": args.reps, "warmup": args.warmup, "pairs": {}}
    try:
        for a, b in (("MicA", "ompA"), ("OxyS", "fhlA")):
            s1, s2 = seqs[a], seqs[b]
            pair = [(s1, s2)]
            cons = [("x" * 5 + "." * (len(s1) - 5), "x" * 5 + "." * (len(s2) - 5))]
            energies = [(shape_deigan(reactivities(len(s1))), shape_deigan(reactivities(len(s2))))]
            batches = {"plain": stage.batch(pair, o), "constrained": stage.batch(pair, o, cons),
                       "shaped": stage.batch(pair, o, None, energies), "both": stage.batch(pair, o, cons, energies)}
            host = {k: [] for k in batches}
            ev = {k: [] for k in batches}
            for rep in range(args.warmup + args.reps):
                for k, bt in batches.items():
                    t0 = time.perf_counter()
                    bt.run()
                    bt.sync()
                    t1 = time.perf_counter()
                    if rep >= args.warmup:
                        host[k].append((t1 - t0) * 1e3)
                        ev[k].append(stage.last_timing().ms_total)
            for bt in batches.values():
                bt.close()
            out["pairs"][f"{a}x{b}"] = {k: {"host_ms_median": statistics.median(host[k]),
                                             "event_ms_median": statistics.median(ev[k]),
                                             "host_ms_min": min(host[k]), "host_ms_max": max(host[k])}
                                         for k in batches}
    finally:
        stage.close()
    text = json.dumps(out)
    print(text)
    if args.out:
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
