#!/usr/bin/env python3
"""Samples per second of the general kernel's sampling phase (the DESIGN section 6 table).

    python tools/sample_latency.py [--reps 30] [--warmup 5] [--out FILE]

Three cases, each a device batch created once and run with rp_batch_run + rp_batch_sync, sampled and unsampled
alternated rep by rep, median of --reps after --warmup:
  mica_ompa   MicA x ompA, 1000 samples of each of its three problems
  long_pair   one random 1000 x 500 pair (the cluster route), 1000 co-fold samples
  batch100    100 MicA x ompA pairs, 100 samples of each problem
Two clocks: the host clock around run + sync, and the library's CUDA events around the launches (rp_timing::ms_total).
A sampled batch runs every sampled problem on the general kernel, so the difference to the unsampled batch (band
kernels where they apply) is route plus sampling.  The oracle sampler (tests/cpp/oracle_sample.c, one CPU thread) is
timed on the MicA x ompA case and on 100 samples of the long pair's co-fold.  The card's name, power limit and
maximum SM clock are read in the same run.  Prints one JSON object (and writes it to --out).  Needs a GPU.
"""
import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

from ractip_b200 import ProbabilityStage, default_model, default_opts  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True)
    return q.stdout.strip()


def oracle_sampler(tmp):
    so = Path(tmp) / "liboracle_sample.so"
    subprocess.run(["gcc", "-O3", "-fPIC", "-shared", "-I", str(ROOT / "include"), "-I", str(ROOT / "ractip_b200" / "csrc"),
                    str(ROOT / "tests" / "cpp" / "oracle_sample.c"), "-o", str(so), "-lm"], check=True)
    lib = C.CDLL(str(so))
    vp, i = C.c_void_p, C.c_int
    lib.orc_params_new.restype = vp
    lib.orc_params_new.argtypes = [vp]
    lib.orc_sample_soft.restype = i
    lib.orc_sample_soft.argtypes = [vp, C.c_char_p, i, i, vp, vp, C.c_uint64, i, i, i, i, vp]
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    seqs = json.loads((ROOT / "tests" / "golden" / "bundled_pairs.json").read_text())["sequences"]
    mo = (seqs["MicA"], seqs["ompA"])
    rng = np.random.default_rng(5)
    long_pair = ("".join("ACGU"[x] for x in rng.integers(0, 4, 1000)), "".join("ACGU"[x] for x in rng.integers(0, 4, 500)))
    cases = {"mica_ompa": ([mo], 1000, ("s1", "s2", "co")),
             "long_pair": ([long_pair], 1000, ("co",)),
             "batch100": ([mo] * 100, 100, ("s1", "s2", "co"))}
    out = {"card": card(), "reps": args.reps, "warmup": args.warmup, "cases": {}}
    stage = ProbabilityStage()
    o = default_opts()
    try:
        for name, (pairs, num, problems) in cases.items():
            batches = {"unsampled": stage.batch(pairs, o),
                       "sampled": stage.batch(pairs, o, samples=num, sample_seed=1, sample_problems=problems)}
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
            drawn = sum(num for a, b in pairs for p in problems if p == "s1" or b)
            res = {k: {"host_ms_median": statistics.median(host[k]), "event_ms_median": statistics.median(ev[k]),
                       "host_ms_min": min(host[k]), "host_ms_max": max(host[k])} for k in batches}
            res["samples"] = drawn
            res["samples_per_s_host"] = drawn / (res["sampled"]["host_ms_median"] * 1e-3)
            out["cases"][name] = res
    finally:
        stage.close()
    # the oracle sampler on one CPU thread: tables plus samples
    with tempfile.TemporaryDirectory() as tmp:
        lib = oracle_sampler(tmp)
        m = default_model()
        P = lib.orc_params_new(C.addressof(m))
        for name, pairs_probs, num in (("mica_ompa", ((mo[0], 0, 0), (mo[1], 0, 1), (mo[0] + mo[1], len(mo[0]) + 1, 2)), 1000),
                                       ("long_pair", ((long_pair[0] + long_pair[1], len(long_pair[0]) + 1, 2),), 100)):
            t0 = time.perf_counter()
            for seq, cp, kind in pairs_probs:
                buf = np.zeros((num, len(seq)), dtype=np.int16)
                assert lib.orc_sample_soft(P, seq.encode(), len(seq), cp, None, None, 1, 0, kind, 0, num,
                                           buf.ctypes.data) == 0
            dt = time.perf_counter() - t0
            out["cases"][name]["oracle_cpu"] = {"samples": num * len(pairs_probs), "s": dt,
                                                "samples_per_s": num * len(pairs_probs) / dt}
    text = json.dumps(out)
    print(text)
    if args.out:
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
