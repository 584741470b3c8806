#!/usr/bin/env python3
"""Latency of one pair with unpaired pseudo-energies against the same pair without data (the DESIGN section 6 table).

    python tools/unpaired_latency.py [--reps 30] [--warmup 5] [--out FILE]

For MicA x ompA and OxyS x fhlA: a device batch of that one pair, created once, then rp_batch_run + rp_batch_sync,
median of --reps after --warmup.  Two clocks: the host clock around run + sync, and the library's CUDA events around
the launches (rp_timing::ms_total).  Probed: seeded N(0, 0.5) kcal/mol unpaired pseudo-energies (20 % zero) on both
sequences, which sends all three problems to the general kernel; unprobed: the default plan (band kernels).  The two
are alternated rep by rep.  Prints one JSON object (and writes it to --out).  Needs a GPU: there is no CPU fallback.
"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

from ractip_b200 import ProbabilityStage, default_opts  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    seqs = json.loads((ROOT / "tests" / "golden" / "bundled_pairs.json").read_text())["sequences"]
    rng = np.random.default_rng(7)

    def energies(n):
        u = rng.normal(0, 0.5, n)
        u[rng.random(n) < 0.2] = 0.0
        return u

    stage = ProbabilityStage()
    o = default_opts()
    out = {"card": card(), "reps": args.reps, "warmup": args.warmup, "pairs": {}}
    try:
        for a, b in (("MicA", "ompA"), ("OxyS", "fhlA")):
            pair = [(seqs[a], seqs[b])]
            ue = [(energies(len(seqs[a])), energies(len(seqs[b])))]
            batches = {"unprobed": stage.batch(pair, o), "probed": stage.batch(pair, o, unpaired_energies=ue)}
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
