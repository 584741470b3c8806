"""The batch planner (ractip_b200/csrc/plan.cpp) on a CPU: which kernel runs each problem, the queues, the
unpaired-window mode, the launch shapes and the split fetch, for the batches the benchmark and the GPU tests run.
Device facts are those of a B200: 148 SMs, 232448 B of opt-in shared memory, general kernel 2 CTAs per SM
(64-register build) / 1 (128-register build), band classes L / S 1 / 2, unstru_kernel 1."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

from ractip_b200._lib import RpOpts, RpPair

ROOT = Path(__file__).resolve().parent.parent
JOB_UNPAIRED = 0x40000000
B200 = dict(sm_count=148, smem_optin=232448, ctas_per_sm=2, ctas_per_sm1=1, up_ctas_per_sm=1, ws_bytes=0,
            occ_l=1, occ_s=2, memory=170 << 30)
SCALARS = ["n_probs", "n_order", "n_band0", "n_band1", "n_general", "n_mcc", "n_duplex", "up_mode", "n_defer",
           "mcc_minb", "grid", "cluster", "band_grid0", "band_grid1", "up_grid", "dom_kind", "split_fetch",
           "n_sect_long", "n_sect_short", "memory_calls", "total_floats", "ws_doubles", "defer_slot", "slot_doubles"]
MICA, OMPA = 72, 137   # bundled MicA x ompA: a shuffle keeps the lengths, and the plan depends on nothing else


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = tmp_path_factory.mktemp("plan") / "libplan_shim.so"
    csrc = ROOT / "ractip_b200" / "csrc"
    subprocess.run(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", str(ROOT / "include"), "-I", str(csrc),
                    str(csrc / "plan.cpp"), str(ROOT / "tests" / "cpp" / "plan_shim.cpp"), "-o", str(so)],
                   check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    lib = C.CDLL(str(so))
    lib.plan_shim.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    lib.plan_shim.restype = C.c_int
    lib.rp_kernel_plan.argtypes = [C.c_int, C.c_size_t, C.c_void_p]
    lib.rp_kernel_plan.restype = C.c_int
    return lib


def opts(duplex=0):
    return RpOpts(max_w=15, min_w=5, th_ss=0.5, th_hy=0.1, th_ac=0.003, use_pf_duplex=duplex)


def seq(n):
    return "ACGU" * (n // 4) + "ACGU"[:n % 4]


def plan(shim, lengths, o=None, band=True, long_n=700, cluster=-1, split_fetch=True, **facts):
    f = dict(B200, **facts)
    strs = [(seq(a).encode(), seq(b).encode()) for a, b in lengths]
    pairs = (RpPair * max(1, len(strs)))()
    for k, (a, b) in enumerate(strs):
        pairs[k].s1, pairs[k].n1, pairs[k].s2, pairs[k].n2 = a, len(a), b or None, len(b)
    fv = np.array([f[k] for k in ("sm_count", "smem_optin", "ctas_per_sm", "ctas_per_sm1", "up_ctas_per_sm",
                                  "ws_bytes", "occ_l", "occ_s", "memory")], dtype=np.int64)
    sv = np.array([int(band), long_n, cluster, int(split_fetch)], dtype=np.int32)
    out = np.zeros(32 + 20 * len(strs) + 64, dtype=np.int64)
    o = o or opts()
    rc = shim.plan_shim(pairs, len(strs), C.byref(o), fv.ctypes.data, sv.ctypes.data, out.ctypes.data, out.size)
    assert rc == 0
    p = dict(zip(SCALARS, out[:len(SCALARS)].tolist()))
    x = 32
    p["order"] = out[x:x + p["n_order"]].tolist()
    x += p["n_order"]
    probs = out[x:x + 4 * p["n_probs"]].reshape(-1, 4)
    p["kind"], p["n"], p["defer_up"], p["ws_off"] = (probs[:, k].tolist() for k in range(4))
    x += 4 * p["n_probs"]
    sects = out[x:x + 2 * (p["n_sect_long"] + p["n_sect_short"])].reshape(-1, 2).tolist()
    p["sect_long"], p["sect_short"] = sects[:p["n_sect_long"]], sects[p["n_sect_long"]:]
    return p


def shuffles(n):
    return [(MICA, OMPA)] * n


def segments(p):
    """The queue as [class L, class S, general, unstru_kernel]."""
    a, b, g = p["n_band0"], p["n_band1"], p["n_general"]
    o = p["order"]
    return o[:a], o[a:a + b], o[a + b:a + b + g], o[a + b + g:]


def test_threshold_of_the_long_build(shim):
    assert shim.rp_kernel_plan(699, 0, None) == 2   # RP_KERNEL_GENERAL
    assert shim.rp_kernel_plan(700, 0, None) == 3   # RP_KERNEL_GENERAL_WIDE
    assert [shim.rp_kernel_plan(n, 0, None) for n in (95, 96, 223, 224)] == [1, 0, 0, 2]


def test_1000_shuffles_defer_the_pass_to_its_own_launch(shim):
    n = 1000
    p = plan(shim, shuffles(n))
    ompa, cofold, mica = [3 * k + 1 for k in range(n)], [3 * k + 2 for k in range(n)], [3 * k for k in range(n)]
    cl, cs, gen, up = segments(p)
    assert (p["n_band0"], p["n_band1"], p["n_general"], p["n_mcc"]) == (2 * n, n, 0, 0)
    assert cl == ompa + cofold and cs == mica and gen == []
    assert p["up_mode"] == 1 and p["n_defer"] == 2 * n
    assert up == ompa + mica   # longest first
    slot = p["defer_slot"]
    assert [p["ws_off"][k] for k in ompa + mica] == [k * slot for k in range(2 * n)]
    assert all(p["ws_off"][k] == -1 and not p["defer_up"][k] for k in cofold)
    assert (p["band_grid0"], p["band_grid1"], p["up_grid"], p["grid"]) == (148, 296, 148, 0)
    assert p["dom_kind"] == 0 and p["memory_calls"] == 1
    # split fetch: the long class writes bp2 and hp, the short class bp1, and the deferred launch up1 + up2
    bp1, bp2, up1, up2 = (MICA + 1) * (MICA + 2) // 2, (OMPA + 1) * (OMPA + 2) // 2, MICA * 15, OMPA * 15
    assert p["split_fetch"] == 1
    assert p["sect_long"] == [[bp1, bp2], [bp1 + bp2 + up1 + up2, (MICA + 1) * (OMPA + 1)]]
    assert p["sect_short"] == [[0, bp1], [bp1 + bp2, up1 + up2]]
    assert not plan(shim, shuffles(n), split_fetch=False)["split_fetch"]


def test_250_shuffles_run_the_pass_as_jobs_of_the_band_kernel(shim):
    n = 250
    p = plan(shim, shuffles(n))
    ompa, cofold, mica = [3 * k + 1 for k in range(n)], [3 * k + 2 for k in range(n)], [3 * k for k in range(n)]
    assert p["up_mode"] == 2 and p["n_defer"] == 2 * n
    cl, cs, gen, up = segments(p)
    # per class: the wavefronts with a dependent job, the others, then the unpaired-window jobs
    assert cl == ompa + cofold + [k | JOB_UNPAIRED for k in ompa]
    assert cs == mica + [k | JOB_UNPAIRED for k in mica]
    assert gen == [] and up == []
    assert (p["band_grid0"], p["band_grid1"], p["dom_kind"]) == (148, 296, 0)
    assert all(p["defer_up"][k] for k in ompa + mica)


def test_125_shuffles_fuse_the_pass(shim):
    n = 125
    p = plan(shim, shuffles(n))
    assert p["up_mode"] == 0 and p["n_defer"] == 0 and p["memory_calls"] == 0
    assert not any(x & JOB_UNPAIRED for x in p["order"]) and not any(p["defer_up"])
    assert p["order"] == [3 * k + 1 for k in range(n)] + [3 * k + 2 for k in range(n)] + [3 * k for k in range(n)]


@pytest.mark.parametrize("n", [1000, 250])
def test_no_room_for_private_workspaces_fuses_the_pass(shim, n):
    p = plan(shim, shuffles(n), memory=1 << 30)
    assert p["up_mode"] == 0 and p["n_defer"] == 0 and not any(p["defer_up"]) and p["ws_off"] == [-1] * 3 * n
    assert p["order"] == [3 * k + 1 for k in range(n)] + [3 * k + 2 for k in range(n)] + [3 * k for k in range(n)]
    assert p["memory_calls"] == 1
    # a workspace already large enough is not asked about
    held = plan(shim, shuffles(n), memory=1 << 30, ws_bytes=1 << 40)
    assert held["up_mode"] > 0 and held["memory_calls"] == 0


def test_one_long_pair_runs_on_16_cta_clusters(shim):
    p = plan(shim, [(1000, 500)])
    assert (p["n_band0"], p["n_band1"], p["n_general"], p["n_mcc"]) == (0, 0, 3, 3)
    assert p["order"] == [2, 0, 1]
    assert (p["mcc_minb"], p["cluster"], p["grid"], p["dom_kind"]) == (1, 16, 3, 2)


def test_20_mid_length_pairs_run_on_8_cta_clusters(shim):
    p = plan(shim, [(400, 300)] * 20)
    assert (p["n_general"], p["mcc_minb"], p["cluster"], p["grid"]) == (60, 1, 8, 60)


def test_148_long_pairs_run_one_cta_per_problem(shim):
    p = plan(shim, [(1000, 500)] * 148)
    assert (p["n_mcc"], p["mcc_minb"], p["cluster"], p["grid"], p["dom_kind"]) == (444, 1, 0, 148, 2)
    assert p["memory_calls"] == 1 and p["ws_doubles"] == 148 * p["slot_doubles"]
    # fewer, fatter slots when the device is short of memory: 70 % of what is available
    small = plan(shim, [(1000, 500)] * 148, memory=50 << 30)
    assert small["grid"] == (50 << 30) // 10 * 7 // (8 * p["slot_doubles"])
    assert plan(shim, [(1000, 500)] * 148, ws_bytes=1 << 40)["memory_calls"] == 0


def test_band_off_routes_everything_to_the_general_kernel(shim):
    """RP_BAND=0, as test_band_and_general_kernels_agree sets it (6 shuffles + CopA x CopT)."""
    lengths = shuffles(6) + [(70, 70)]
    assert plan(shim, lengths)["n_general"] == 0
    p = plan(shim, lengths, band=False)
    assert (p["n_band0"], p["n_band1"], p["n_general"], p["n_mcc"], p["up_mode"]) == (0, 0, 21, 21, 0)
    assert (p["mcc_minb"], p["cluster"], p["split_fetch"], p["dom_kind"]) == (2, 8, 0, 2)


@pytest.mark.parametrize("long_n,cluster,minb,g", [(216, -1, 1, 16), (700, -1, 2, 16), (224, 0, 1, 0), (224, 8, 1, 8),
                                                   (224, 16, 1, 16), (100000, 0, 2, 0)])
def test_forced_builds_and_cluster_sizes(shim, long_n, cluster, minb, g):
    """RP_MCC_LONG_N and RP_CLUSTER as test_wide_split_sum_bands and test_multi_cta_wavefront_matches_oracle set them."""
    p = plan(shim, [(300, 130), (230, 261), (40, 610)], long_n=long_n, cluster=cluster)
    assert (p["mcc_minb"], p["cluster"]) == (minb, g)


def test_duplex_lone_sequence_and_empty_batch(shim):
    p = plan(shim, [(35, 35), (72, 137), (70, 70)], opts(duplex=1))
    assert p["n_duplex"] == 3 and p["n_mcc"] == 0 and p["n_general"] == 3
    assert [p["kind"][k] for k in p["order"][-3:]] == [2, 2, 2]   # the duplex problems, last
    assert p["grid"] == 3 and p["cluster"] == 0 and p["slot_doubles"] == 2 * (72 + 2) * (137 + 2)
    lone = plan(shim, [(50, 0)])
    assert lone["n_probs"] == 3 and lone["order"] == [0] and lone["n"] == [50, 0, 0]
    empty = plan(shim, [])
    assert (empty["n_probs"], empty["n_order"], empty["dom_kind"], empty["memory_calls"]) == (0, 0, -1, 0)
