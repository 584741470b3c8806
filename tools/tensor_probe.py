#!/usr/bin/env python3
"""Timing of the device exits to PyTorch on the z-score shuffle batch (MicA x ompA, --zscore=12, seed 1).

    python tools/tensor_probe.py [--num 1000] [--reps 10] [--kernel-reps 200] [--out FILE]

* square_kernel: CUDA events around --kernel-reps back-to-back rp_batch_square_device calls (one launch each) after
  warm-up, five such windows; the batch's outputs (102 KB per pair) and the square tensors (150 KB per pair) together
  exceed the 126 MB L2 at 1000 pairs, so every window streams from and to HBM.
* the two ways to get the square tensors to torch, alternated rep by rep, host clock around work that ends in a device
  synchronise: (a) run + tensors(); (b) run + fetch_dense() + per-pair slicing and padding on the host + upload.
  Each is timed whole (run and exit overlap as they can) and exit only (after a synchronised run).
Prints one JSON object (and writes it to --out).  Needs a GPU: there is no CPU fallback.
"""
import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from ractip_b200 import ProbabilityStage, bp_offsets, default_opts, zscore_shuffles  # noqa: E402
from ractip_b200.stage import SQUARE_KEYS  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], stdout=subprocess.PIPE, text=True)
    return q.stdout.strip()


def host_square(b, flat, dev):
    """What a caller does without the device exit: slice the fetched block pair by pair, unpack the packed upper
    triangles into padded symmetric matrices, upload."""
    lay = b.square_layout()
    B, N1, N2, W = lay.B, lay.N1, lay.N2, lay.W
    out = {"bp1": np.zeros((B, N1 + 1, N1 + 1), np.float32), "bp2": np.zeros((B, N2 + 1, N2 + 1), np.float32),
           "up1": np.zeros((B, N1, W), np.float32), "up2": np.zeros((B, N2, W), np.float32),
           "hp": np.zeros((B, N1 + 1, N2 + 1), np.float32)}
    tri = {}
    for k, r in enumerate(b.split_dense(flat)):
        for key, bp, off in (("bp1", r.bp1, r.offset1), ("bp2", r.bp2, r.offset2)):
            n = len(off) - 1
            if n not in tri:
                i, j = np.triu_indices(n + 1, 1)
                i, j = i[i >= 1], j[i >= 1]
                tri[n] = (i, j, bp_offsets(n)[i].astype(np.int64) + j)
            i, j, idx = tri[n]
            v = bp[idx]
            out[key][k, i, j] = v
            out[key][k, j, i] = v
        out["up1"][k, :r.up1.shape[0]] = r.up1
        out["up2"][k, :r.up2.shape[0]] = r.up2
        if r.hp.shape[1] > 1:
            out["hp"][k, :r.hp.shape[0], :r.hp.shape[1]] = r.hp
    return {k: torch.from_numpy(v).to(dev) for k, v in out.items()}


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--num", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--kernel-reps", type=int, default=200)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tensor_probe.py: no CUDA device")
    seqs = json.loads((ROOT / "tests" / "golden" / "bundled_pairs.json").read_text())["sequences"]
    r1, r2 = zscore_shuffles(seqs["MicA"], seqs["ompA"], args.num, 1)
    st = ProbabilityStage(device=torch.cuda.current_device())
    dev = st.torch_device()
    b = st.batch(list(zip(r1, r2)), default_opts())
    b.run()
    lay = b.square_layout()
    res = {"card": card(), "pairs": args.num, "n1": len(seqs["MicA"]), "n2": len(seqs["ompA"]),
           "dense_bytes": b.total_floats * 4,
           "square_bytes": 4 * (lay.n_bp1 + lay.n_bp2 + lay.n_up1 + lay.n_up2 + lay.n_hp)}

    # the two exits agree bit for bit
    t = b.tensors()
    h = host_square(b, b.fetch_dense()[:b.total_floats], dev)
    torch.cuda.synchronize()
    res["bitwise_equal"] = all(torch.equal(t[k].view(torch.int32), h[k].view(torch.int32)) for k in SQUARE_KEYS)

    # square_kernel by itself
    ptrs = [C.c_void_p(t[k].data_ptr() if t[k].numel() else None) for k in SQUARE_KEYS]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    windows = []
    with st._torch_stream():
        for _ in range(20):
            st._check(b.lib.rp_batch_square_device(b.handle, *ptrs))
        for _ in range(5):
            e0.record()
            for _ in range(args.kernel_reps):
                st._check(b.lib.rp_batch_square_device(b.handle, *ptrs))
            e1.record()
            e1.synchronize()
            windows.append(e0.elapsed_time(e1) / args.kernel_reps)
    ms = statistics.median(windows)
    res["square_kernel_ms"] = spread(windows)
    # least traffic: every output element written once, every dense float of the five sections read once
    res["square_kernel_GBps_min_traffic"] = (res["square_bytes"] + res["dense_bytes"]) / (ms * 1e-3) / 1e9

    # whole call and exit only, both ways, alternated
    def exit_a():
        return b.tensors()

    def exit_b():
        return host_square(b, b.fetch_dense()[:b.total_floats], dev)

    whole = {"a": [], "b": []}
    only = {"a": [], "b": []}
    for f in (exit_a, exit_b):   # warm-up
        b.run()
        f()
        torch.cuda.synchronize()
    for _ in range(args.reps):
        for key, f in (("a", exit_a), ("b", exit_b)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            b.run()
            f()
            torch.cuda.synchronize()
            whole[key].append((time.perf_counter() - t0) * 1e3)
            b.run()
            b.sync()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f()
            torch.cuda.synchronize()
            only[key].append((time.perf_counter() - t0) * 1e3)
    res["run_plus_tensors_ms"] = spread(whole["a"])
    res["run_plus_fetch_slice_upload_ms"] = spread(whole["b"])
    res["tensors_only_ms"] = spread(only["a"])
    res["fetch_slice_upload_only_ms"] = spread(only["b"])
    b.close()
    st.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
