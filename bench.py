#!/usr/bin/env python3
"""Benchmark of the probability stage on the --zscore shuffle batch.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload mica_ompa|synthetic] [--num-shuffling 1000] [--scaling strong|weak]
                    [--no-config4] [--no-cpu-baseline] [--dump-outputs DIR]

Metric (BASELINE.json): shuffled pairs / second of the probability stage of
`ractip --zscore=12 --num-shuffling=1000` (per shuffled pair: 2 single-strand
McCaskill inside/outside + 2 unpaired-window passes + 1 two-strand McCaskill).
One "step" = one pass over the whole shuffle batch: kernels + the compaction into the
thresholded variable lists (+ the one all-gather when N > 1).  Prints ONE JSON line.

The headline workload is BASELINE configs[3] (MicA x ompA, 1000 shuffles).  The same run also
measures BASELINE configs[4] (synthetic 1000 x 500 nt pairs, the long-sequence kernels) on a bounded
batch of 148 shuffled pairs per GPU and reports it under the key "config4" with its own roofline,
clocks, e2e and cpu_baseline (--workload synthetic makes it the headline instead, full 1000 pairs).

--impl reference: the reference's probability stage cannot be built here (ViennaRNA absent,
DESIGN.md section 5), so the timed CPU implementation is the oracle port (oracle/) on all host
threads; it does not load the product library.

--dump-outputs DIR: after the timed steps, the thresholded lists x, y, z, v, w of the last step (what a
caller of the timed path receives) go to DIR/<list>.npy, and those of the configs[4] leg to
DIR/config4_<list>.npy: float32 rows (pair index in the batch, i, j, p).  On N GPUs rank 0 writes the lists of
all ranks; with weak scaling the pair index runs over the ranks' batches in rank order.  The inputs depend only
on the arguments, so two builds can be compared output for output.  The legs share 64 MB equally; a leg whose
lists exceed its share is cut to a seeded sample of its pairs.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

METRIC = "shuffled pairs/sec, probability stage of --zscore=12 (McCaskill in/out x2 + unpaired windows x2 + two-strand McCaskill)"
UNIT = "pairs/s"
CONFIG4_PAIRS_PER_GPU = 148      # bounded batch of the configs[4] leg: one two-strand problem per SM
CONFIG4_REF_PAIRS = 8            # ... and of its CPU arm (the port does ~0.5 pairs/s on 16 cores)
DUMP_BYTES = 64 << 20            # --dump-outputs: all legs together


# --------------------------------------------------------------------------- workload
def base_sequences(name: str):
    seqs = json.loads((ROOT / "tests" / "golden" / "bundled_pairs.json").read_text())["sequences"]
    if name == "mica_ompa":
        return seqs["MicA"], seqs["ompA"], "MicA(72) x ompA(137)", "BASELINE configs[3]"
    if name == "synthetic":
        rng = np.random.default_rng(20261018)
        s1 = "".join("ACGU"[x] for x in rng.integers(0, 4, 1000))
        s2 = "".join("ACGU"[x] for x in rng.integers(0, 4, 500))
        return s1, s2, "synthetic 1000 x 500 nt", "BASELINE configs[4]"
    raise SystemExit("unknown workload " + name)


def ref_shuffles(s1: str, s2: str, num: int, seed: int):
    """The shuffles of src/ractip.cpp:1636-1643 from the REFERENCE's own src/ushuffle.c (oracle/_ref, built by
    oracle/Makefile) on glibc random(): srandom(seed); per iteration shuffle(s1, k=2) then shuffle(s2, k=2)."""
    so = ROOT / "oracle" / "_ref" / "libushuffle_ref.so"
    if not so.exists():
        return None
    ref, libc = C.CDLL(str(so)), C.CDLL(None)
    libc.srandom(C.c_uint(seed))
    ref.set_randfunc(C.cast(libc.random, C.c_void_p))
    b1, b2 = C.create_string_buffer(len(s1) + 1), C.create_string_buffer(len(s2) + 1)
    out = []
    for _ in range(num):
        ref.shuffle(s1.encode(), b1, len(s1), 2)
        ref.shuffle(s2.encode(), b2, len(s2), 2)
        out.append((b1.raw[:len(s1)].decode(), b2.raw[:len(s2)].decode()))
    return out


def make_workload(name: str, num: int, seed: int, impl: str):
    s1, s2, what, cfg = base_sequences(name)
    pairs = ref_shuffles(s1, s2, num, seed) if impl == "reference" else None
    gen = "src/ushuffle.c (oracle/_ref) + glibc random()"
    if pairs is None:
        from ractip_b200 import zscore_shuffles   # bit-exact restatement of the same generator (tests/test_shuffle.py)
        r1, r2 = zscore_shuffles(s1, s2, num, seed, mode=12, k=2)
        pairs, gen = list(zip(r1, r2)), "rp_zscore_shuffles"
    desc = f"{what}, --zscore=12 --num-shuffling={num} --seed={seed} ({cfg})"
    data = ("dinucleotide shuffles (uShuffle k=2, seed %d) of the bundled MicA / ompA sequences" % seed if name == "mica_ompa"
            else "synthetic: dinucleotide shuffles (seed %d) of one i.i.d. uniform 1000-nt and one 500-nt sequence" % seed)
    return pairs, desc, data, gen


def load_model_fixture():
    """The default integer energy model (BL* + residual Turner-2004 tables) from the committed fixture, so that
    the reference arm does not need the product library (tests/golden/gen_golden.py writes it)."""
    from ractip_b200._lib import RpModel   # a ctypes struct definition; importing it does not load the .so
    raw = (ROOT / "tests" / "golden" / "default_model.bin").read_bytes()
    assert len(raw) == C.sizeof(RpModel), "tests/golden/default_model.bin is stale: rerun tests/golden/gen_golden.py"
    return RpModel.from_buffer_copy(raw)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                clk, mxc = float(parts[0]), float(parts[1])
            except ValueError:
                continue
            mx = mxc
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk)
                for nm, val in zip(names, parts[3:7]):
                    if val == "Active":
                        reasons.add(nm)
        if not sm:
            sm = [float(l.split(",")[0]) for _, l in self.rows[-3:] if l.split(",")[0].strip().replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------- CPU oracle timing
def cpu_pairs_per_second(pairs, threads: int, model):
    """Times the CPU restatement (oracle/, kind 'port') on `pairs` with `threads` host threads."""
    from oracle.oracle import Oracle
    o = Oracle(model)
    todo = list(pairs)
    lock = threading.Lock()

    def work():
        while True:
            with lock:
                if not todo:
                    return
                a, b = todo.pop()
            o.rnafold(a, 15)
            o.rnafold(b, 15)
            o.rnaduplex(a, b, 0.1)

    t0 = time.perf_counter()
    ths = [threading.Thread(target=work) for _ in range(threads)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return len(pairs) / dt, dt


def cpu_baseline(pairs, model, sample_n: int, single_n: int, e2e_value=None):
    cores = os.cpu_count() or 1
    v_all, dt_all = cpu_pairs_per_second(pairs[:sample_n], cores, model)
    v_1, dt_1 = cpu_pairs_per_second(pairs[:single_n], 1, model)
    out = {"value": v_all, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"first {sample_n} shuffled pairs of the workload on {cores} threads ({dt_all:.1f} s)",
           "single_thread_value": v_1,
           "single_thread_sample": f"first {single_n} pairs on 1 thread ({dt_1:.1f} s); the reference runs single-threaded (src/ractip.cpp:1494)"}
    if e2e_value:
        out["e2e_over_all_cores"] = e2e_value / v_all
        out["e2e_over_single_thread"] = e2e_value / v_1
    return out


def run_reference(args, rank: int, world: int):
    """The CPU arm: same workload, config keys and pairs per step as ours for configs[3]; the configs[4] leg is a
    bounded sample.  Loads oracle/ (and oracle/_ref for the shuffles), never the product library."""
    if rank != 0:
        return
    model = load_model_fixture()
    cores = os.cpu_count() or 1

    def arm(workload, per_step, steps, warmup):
        pairs, desc, data, gen = make_workload(workload, args.num_shuffling, args.seed, "reference")
        for _ in range(min(warmup, 1)):
            cpu_pairs_per_second(pairs[:cores], cores, model)
        tot_pairs, tot_t = 0, 0.0
        for s in range(steps):
            sample = [pairs[(s * per_step + k) % len(pairs)] for k in range(per_step)]
            _, dt = cpu_pairs_per_second(sample, cores, model)
            tot_pairs += len(sample)
            tot_t += dt
        v = tot_pairs / tot_t
        return {
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": 1e3 * tot_t / steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": data,
            "config": {"workload": desc, "pairs_per_step": per_step, "sharding": "none (host threads over pairs)",
                       "collective": "none", "l2": "n/a (CPU)", "kernels": "oracle/rp_oracle.c (CPU port of the path)",
                       "shuffles": gen},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{tot_pairs} shuffled pairs of the workload, {cores} threads over pairs "
                                       "(the reference itself is single-threaded, src/ractip.cpp:1494)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }

    if args.workload == "mica_ompa":
        line = arm("mica_ompa", args.num_shuffling, args.steps, args.warmup)
        if not args.no_config4:
            c4 = arm("synthetic", CONFIG4_REF_PAIRS, args.steps, args.warmup)
            line["config4"] = {k: c4[k] for k in ("value", "unit", "steps", "ms_per_step", "config", "cpu_baseline", "e2e", "data")}
    else:
        line = arm("synthetic", max(2, cores // 4), args.steps, args.warmup)
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- our arm
def traffic_record(workload: str):
    """DRAM bytes per launch of the dominant kernel, with the ncu capture it was read from (profiles/traffic.json)."""
    tf = ROOT / "profiles" / "traffic.json"
    if not tf.exists():
        return None, None
    try:
        rec = json.loads(tf.read_text()).get(workload)
    except Exception:
        return None, None
    if isinstance(rec, dict):
        return rec.get("bytes_per_launch"), {k: v for k, v in rec.items() if k != "bytes_per_launch"}
    return rec, None


def step_lists(plan, pairs_all, opts, buf, world: int, weak: bool):
    """PairRecords of every pair of a step from the host copy of the gathered buffer (of `local` when N = 1), in batch
    order.  With weak scaling each rank ran a batch of its own, laid out by its own plan at the start of its
    equally sized slot; the batches follow one another in rank order."""
    if not weak:
        return plan.unpack(buf)
    from ractip_b200.dist import ShardPlan
    slots = buf.reshape(world, -1)
    out = []
    for r in range(world):
        own = ShardPlan(pairs_all[r], opts, 0, 1)
        out += own.unpack(slots[r][:own.nbytes])
    return out


def dump_outputs(out_dir: Path, legs):
    """--dump-outputs: legs = [(file prefix, PairRecords of every pair in batch order)]."""
    out_dir.mkdir(parents=True, exist_ok=True)
    for prefix, recs in legs:
        assert len(recs) < 1 << 24, "pair indices must stay exact in float32"
        nbytes = np.array([sum(len(getattr(r, name)) for name in "xyzvw") * 16 for r in recs])
        order = np.random.default_rng(0).permutation(len(recs))
        keep = np.sort(order[:np.searchsorted(np.cumsum(nbytes[order]), DUMP_BYTES // len(legs), side="right")])
        for name in "xyzvw":
            lists = [getattr(recs[k], name) for k in keep]
            rows = [np.column_stack([np.full(len(a), k), a["i"], a["j"], a["p"]]) for k, a in zip(keep, lists)]
            np.save(out_dir / f"{prefix}{name}.npy",
                    np.concatenate(rows).astype(np.float32) if rows else np.zeros((0, 4), dtype=np.float32))


def measure(args, stage, workload, pairs_all, desc, data, rank, world, local_rank, steps, warmup, scaling, dev, stream,
            cpu_sample, with_cpu, dump=False):
    """One workload through the three measurements: device-resident step ("value"), end to end through the C ABI
    with host buffers ("e2e"), roofline of the kernels and the CPU port beside it (rank 0, N = 1).  dump: rank 0 also
    returns the lists of the last timed step under "outputs"."""
    import torch
    import torch.distributed as dist

    from ractip_b200 import default_opts
    from ractip_b200._lib import RpPair
    from ractip_b200.dist import ShardPlan
    lib = stage.lib
    opts = default_opts()
    if scaling == "weak" and world > 1:
        mine_idx = None
        mine = pairs_all[rank]          # pairs_all: one list per rank
        total_pairs = sum(len(p) for p in pairs_all)
        plan = ShardPlan(mine, opts, 0, 1)
        nbytes = torch.tensor([plan.nbytes], device=dev, dtype=torch.int64)
        dist.all_reduce(nbytes, op=dist.ReduceOp.MAX)
        local_bytes = int(nbytes.item())
    else:
        plan = ShardPlan(pairs_all, opts, rank, world)   # interleaved shard of the one shuffle batch
        mine = plan.my_pairs
        total_pairs = len(pairs_all)
        local_bytes = plan.nbytes

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- device-resident batch ("value")
    batch = stage.batch(mine, opts)
    local = torch.zeros(local_bytes, dtype=torch.uint8, device=dev)
    gathered = torch.empty(world * local_bytes, dtype=torch.uint8, device=dev) if world > 1 else None
    cap = plan.rec_bytes // 12

    def step_resident():
        batch.run()
        # thresholded variable lists x, y, z, v, w + counts, written by the compaction kernel into the gather buffer
        base = local.data_ptr()
        stage._check(lib.rp_batch_sparse_device(batch.handle, C.c_void_p(base), cap, C.c_void_p(0), 0,
                                                C.c_void_p(base + plan.rec_bytes)))
        if world > 1:
            dist.all_gather_into_tensor(gathered, local)   # the single collective of the path

    for _ in range(warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    time.sleep(0.25)
    t_wall0 = time.time()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern_ms, dom_ms, launches = [], [], 0
    ev0.record(stream)
    for _ in range(steps):
        step_resident()
        if world == 1:
            t = stage.last_timing()      # CUDA events around the kernels on their stream
            kern_ms.append(t.ms_total)
            dom_ms.append(t.ms_dominant)
            launches += t.kernel_launches
        else:
            launches += 4                # two band launches (or one general), the compaction, the collective
    ev1.record(stream)
    barrier()
    t_wall1 = time.time()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop(t_wall0, t_wall1)
    if world > 1:
        tmax = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item())
    ms_per_step = ms / steps
    value = total_pairs / (ms_per_step * 1e-3)

    # the timed path must have produced real data: this rank's lists equal a fresh rp_run_sparse of its shard
    chk = stage.run_sparse(mine[:3], opts)
    if scaling == "weak" and world > 1:
        mine_plan, my_buf = plan, local.cpu().numpy()
    else:
        mine_plan, my_buf = plan, (gathered.cpu().numpy().reshape(world, -1)[rank] if world > 1 else local.cpu().numpy())
    recs = mine_plan.rec_view(my_buf)
    cnt = my_buf[plan.rec_bytes:plan.rec_bytes + 24 * len(mine)].view(np.int32).reshape(-1, 6)
    lay = mine_plan.layouts[0 if (scaling == "weak" and world > 1) else rank]
    for k, c in enumerate(chk):
        S = lay[k]
        assert not cnt[k][3], "record capacity exceeded"
        for name, off, n_k, want in (("x", S.x, cnt[k][0], c.x), ("z", S.z, cnt[k][2], c.z), ("v", S.v, cnt[k][4], c.v)):
            assert recs[off:off + int(n_k)].tolist() == want.tolist(), f"gathered {name} records differ"
    if world > 1 and scaling != "weak":
        g = gathered.cpu().numpy().reshape(world, -1)
        for r in range(world):
            cr = g[r][plan.rec_bytes:plan.rec_bytes + 24 * len(plan.shards[r])].view(np.int32).reshape(-1, 6)
            assert cr[:, :3].sum() > 0, f"rank {r} gathered nothing"
    outputs = None
    if dump and rank == 0:
        outputs = step_lists(plan, pairs_all, opts, (gathered if world > 1 else local).cpu().numpy(), world,
                             scaling == "weak" and world > 1)

    # ---------------- end to end through the C ABI with host buffers
    n = len(mine)
    arr = (RpPair * max(n, 1))()
    keep = []
    for k, (a, b) in enumerate(mine):
        ba, bb = a.encode(), b.encode()
        keep.append((ba, bb))
        arr[k].s1, arr[k].n1, arr[k].s2, arr[k].n2 = ba, len(ba), bb, len(bb)
    out_bytes = batch.total_floats * 4
    pin = lib.rp_host_alloc(max(out_bytes, 4))
    pin_recs = lib.rp_host_alloc(max(batch.total_recs * 12, 4))
    pin_cnt = lib.rp_host_alloc(max(n * 24, 24))
    # encoded sequences + 3 problem descriptors (72 B) + 3 queue entries per pair
    h2d_bytes = sum(2 * (len(a) + len(b)) + 4 for a, b in mine) + 3 * n * 72 + 3 * n * 4

    def e2e_dense():
        stage._check(lib.rp_run_dense(stage.ctx, arr, n, C.byref(opts), C.c_void_p(pin), batch.total_floats))

    def e2e_sparse():
        stage._check(lib.rp_run_sparse(stage.ctx, arr, n, C.byref(opts), C.c_void_p(pin_recs), batch.total_recs,
                                       C.c_void_p(0), 0, C.c_void_p(pin_cnt)))

    def time_e2e(fn):
        for _ in range(max(1, warmup - 1)):
            fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(steps):
            fn()
        b.record(stream)
        barrier()
        t = a.elapsed_time(b)
        if world > 1:
            tm = torch.tensor([t], device=dev, dtype=torch.float64)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            t = float(tm.item())
        return total_pairs / (t / steps * 1e-3)

    e2e_d = time_e2e(e2e_dense)
    e2e_s = time_e2e(e2e_sparse)

    # ---------------- roofline of the kernels + CPU baseline (rank 0, N=1)
    roofline, cpu = None, None
    if world == 1:
        fp64_tf, smem_gbs = stage.measure_peaks()
        batch.run()
        tt = stage.last_timing()
        # The dominant kernel by itself (the contract's roofline): the launch that carries most of the algorithmic flops,
        # CUDA events around it on its stream, its own problems' flops.  Next to it the whole step: ALL kernels of a step
        # (incl. the unpaired-window kernel, whose flops SURVEY 8d does not credit) against all credited flops.
        alg_all = tt.alg_flops
        step_ms = statistics.mean(kern_ms) if kern_ms else tt.ms_total
        alg = tt.alg_flops_dominant
        launch_ms = statistics.mean(dom_ms) if dom_ms and min(dom_ms) > 0 else tt.ms_dominant
        dom_name = {0: "mcc_band_kernel<512,1> (the long band class: the 137-nt strands and the 209-nt two-strand problems)",
                    1: "mcc_band_kernel<256,2> (the short band class)",
                    2: KERNELS[workload][0]}.get(tt.dominant_kind, KERNELS[workload][0])
        achieved = alg / (launch_ms * 1e-3) / 1e12
        achieved_step = alg_all / (step_ms * 1e-3) / 1e12
        traffic, traffic_src = traffic_record(workload)
        if traffic is not None and traffic_src and traffic_src.get("pairs_per_launch"):
            traffic = traffic / traffic_src["pairs_per_launch"] * len(mine)   # scaled to this launch's pair count
        roofline = {
            "bound": "fp64_fma", "kernel": dom_name, "achieved": achieved, "peak": fp64_tf, "unit": "TFLOP/s",
            "frac": achieved / fp64_tf if fp64_tf else None, "traffic": traffic, "traffic_source": traffic_src,
            "alg_flops_per_launch": alg, "launch_ms": launch_ms,
            "whole_step": {"kernels": KERNELS[workload][2], "alg_flops": alg_all, "ms": step_ms, "achieved": achieved_step,
                           "frac": achieved_step / fp64_tf if fp64_tf else None},
            "peak_source": "live fp64-FMA micro-benchmark on this GPU (rp_measure_peaks); "
                           "MEASURED_PEAKS.json holds only HBM/bf16 peaks, which do not bound this path",
            "smem_peak_gbs": smem_gbs,
            "smem_frac_at_16B_per_term": (alg / 2.0 * 16.0 / (launch_ms * 1e-3) / 1e9) / smem_gbs if smem_gbs else None,
        }
        peaks_file = ROOT / "MEASURED_PEAKS.json"
        if peaks_file.exists():
            try:
                hbm = json.loads(peaks_file.read_text()).get("hbm_gbs")
                roofline["hbm_peak_gbs_measured"] = hbm
                if traffic and hbm:
                    roofline["hbm_frac"] = traffic / (launch_ms * 1e-3) / 1e9 / hbm
            except Exception:
                pass
        if with_cpu:
            flat = mine if not (scaling == "weak" and world > 1) else mine
            cpu = cpu_baseline(flat, stage.model, cpu_sample[0], cpu_sample[1], e2e_d)

    res = {
        "value": value, "unit": UNIT, "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step, "scaling": scaling,
        "data": data,
        "config": {"workload": desc, "pairs_per_step": total_pairs,
                   "sharding": (f"shuffles r::{world}" if scaling != "weak" else f"{len(mine)} pairs per rank") if world > 1 else "none",
                   "collective": "one all_gather of the thresholded lists (x, y, z, v, w)" if world > 1 else "none",
                   "l2": "per-step working set (workspace slots of all resident CTAs, > 1 GB) exceeds the 126 MB L2; no flush needed",
                   "kernels": KERNELS[workload][1]},
        "clocks": clocks,
        "e2e": {"value": e2e_d, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes * world,
                "d2h_bytes_per_step": out_bytes * world, "api": "rp_run_dense (reference layouts, pinned host buffer)"},
        "e2e_sparse": {"value": e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes * world,
                       "d2h_bytes_per_step": (batch.total_recs * 12 + n * 24) * world,
                       "api": "rp_run_sparse (thresholded variable lists x, y, z, v, w)"},
        "gpu_launches": launches,
    }
    if roofline:
        res["roofline"] = roofline
    if cpu:
        res["cpu_baseline"] = cpu
    if outputs is not None:
        res["outputs"] = outputs
    lib.rp_host_free(C.c_void_p(pin)); lib.rp_host_free(C.c_void_p(pin_recs)); lib.rp_host_free(C.c_void_p(pin_cnt))
    batch.close()
    return res


def run_ours(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist

    from ractip_b200 import ProbabilityStage, default_model

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the probability stage has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stage = ProbabilityStage(default_model(), device=local_rank)
    # One explicit (non-default) stream carries the kernels, the NCCL collective and the
    # timing events.  (The legacy default stream has handle 0, which rp_set_stream reads as
    # "use the context's own stream": events recorded there would not see the kernels.)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    stage.lib.rp_set_stream(stage.ctx, C.c_void_p(stream.cuda_stream))

    def workload_pairs(name, num, scaling):
        if scaling == "weak" and world > 1:   # fixed per-GPU work: every rank gets its own batch (different seed)
            per = [make_workload(name, num, args.seed + r, "ours") for r in range(world)]
            return [p[0] for p in per], per[0][1], per[0][2]
        pairs, desc, data, _ = make_workload(name, num, args.seed, "ours")
        return pairs, desc, data

    pairs, desc, data = workload_pairs(args.workload, args.num_shuffling, args.scaling)
    cpu_n = (min(args.num_shuffling, 1000), max(1, min(64, args.num_shuffling // 4))) if args.workload == "mica_ompa" \
        else (max(2, (os.cpu_count() or 1) // 4), 1)
    dump = args.dump_outputs is not None
    head = measure(args, stage, args.workload, pairs, desc, data, rank, world, local_rank, args.steps, args.warmup,
                   args.scaling, dev, stream, cpu_n, not args.no_cpu_baseline, dump)
    c4 = None
    if args.workload == "mica_ompa" and not args.no_config4:
        # BASELINE configs[4] in the same run: a bounded batch, fixed work per GPU ("weak")
        per_rank = [make_workload("synthetic", CONFIG4_PAIRS_PER_GPU, args.seed + r, "ours") for r in range(world)]
        p4 = [p[0] for p in per_rank] if world > 1 else per_rank[0][0]
        c4 = measure(args, stage, "synthetic", p4, per_rank[0][1].replace(f"--num-shuffling={CONFIG4_PAIRS_PER_GPU}",
                     f"{CONFIG4_PAIRS_PER_GPU} of the --num-shuffling=1000 shuffles per GPU"), per_rank[0][2], rank, world,
                     local_rank, args.steps, args.warmup, "weak" if world > 1 else "strong", dev, stream,
                     (CONFIG4_REF_PAIRS, 1), not args.no_cpu_baseline, dump)
        if world == 1:
            c4["scaling"] = "weak"
    if dump and rank == 0:
        dump_outputs(Path(args.dump_outputs), [("", head.pop("outputs"))] + ([("config4_", c4.pop("outputs"))] if c4 else []))
    if rank == 0:
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": head["steps"],
                "warmup": head["warmup"], "ms_per_step": head["ms_per_step"], "higher_is_better": True,
                "scaling": head["scaling"], "vs_baseline": None, "dtype": "f64"}
        for k in ("data", "config", "clocks", "e2e", "e2e_sparse", "gpu_launches", "roofline", "cpu_baseline"):
            if k in head:
                line[k] = head[k]
        if c4:
            line["config4"] = c4
            line["gpu_launches"] += c4["gpu_launches"]
        print(json.dumps(line), flush=True)
    stage.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# dominant kernel (roofline) and routing of each workload (rp_kernel_plan / rp_batch_create)
KERNELS = {
    "mica_ompa": ("mcc_band_kernel<512,1>",
                  "mcc_band_kernel<512,1> (n > ~95) + mcc_band_kernel<256,2> (shorter) + unstru_kernel (unpaired windows of a "
                  "large batch) + sparse_kernel; general kernel for n > 223",
                  "mcc_band_kernel<512,1> + <256,2> + unstru_kernel (the unpaired-window pass: no credited flops)"),
    "synthetic": ("mcc_persistent<1,10> (general kernel, HBM tables, 128 registers, split sums in bands of 10 diagonals)",
                  "mcc_persistent<1,10>: one CTA per problem and per SM, 1500 / 1000 / 500-nt problems from one cost-ordered queue; sparse_kernel",
                  "mcc_persistent<1,10> (every pass of a problem in the one launch)"),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="mica_ompa", choices=["mica_ompa", "synthetic"])
    ap.add_argument("--num-shuffling", type=int, default=1000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config4", action="store_true", help="skip the BASELINE configs[4] leg of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the thresholded lists of the last timed step to DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
