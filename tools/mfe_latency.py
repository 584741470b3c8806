#!/usr/bin/env python3
"""Latency of rp_run_mfe, the minimum free energy kernel (the DESIGN section 6 table).

    python tools/mfe_latency.py [--reps 10] [--warmup 2] [--out FILE]

Four cases, each one synchronous rp_run_mfe call (s1, s2 and the s1&s2 co-fold of every pair), median of --reps after
--warmup: MicA x ompA, OxyS x fhlA, one random 1000 x 500 pair (seed 7), and one batch of the eight bundled pairs.
Two clocks: the host clock around the call (copies and planning included) and the library's CUDA events around the
launch (rp_timing::ms_total).  The card's name, power limit and maximum SM clock are read in the same run.  Prints one
JSON object (and writes it to --out).  Needs a GPU.
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

from ractip_b200 import ProbabilityStage, default_model  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    b = json.loads((ROOT / "tests" / "golden" / "bundled_pairs.json").read_text())
    seqs = b["sequences"]
    rng = np.random.default_rng(7)
    rand = lambda n: "".join("ACGU"[x] for x in rng.integers(0, 4, n))
    cases = {
        "mica_ompa": [(seqs["MicA"], seqs["ompA"])],
        "oxys_fhla": [(seqs["OxyS"], seqs["fhlA"])],
        "long_pair": [(rand(1000), rand(500))],
        "bundled8": [(seqs[x], seqs[y]) for x, y in b["pairs"]],
    }
    st = ProbabilityStage(default_model())
    res = {"card": card(), "reps": a.reps, "cases": {}}
    try:
        for name, pairs in cases.items():
            host, dev = [], []
            for r in range(a.warmup + a.reps):
                t0 = time.perf_counter()
                st.mfe(pairs)
                t1 = time.perf_counter()
                if r >= a.warmup:
                    host.append((t1 - t0) * 1e3)
                    dev.append(st.last_timing().ms_total)
            res["cases"][name] = {"pairs": len(pairs), "lengths": [[len(x), len(y)] for x, y in pairs][:8],
                                  "host_ms": statistics.median(host), "kernel_ms": statistics.median(dev)}
    finally:
        st.close()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        Path(a.out).write_text(text)


if __name__ == "__main__":
    main()
