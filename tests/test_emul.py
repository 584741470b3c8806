"""The CUDA kernel's phase functions (ractip_b200/csrc/mcc_core.h + mcc_driver.h), compiled
for the host and run thread after thread, against the oracle.  This checks the kernel LOGIC
on a CPU-only box; the gpu-marked tests check the real kernel."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from conftest import rand_seq


@pytest.mark.parametrize("T", [33, 64, 256])
def test_emulated_linear_matches_oracle(emul, oracle, T):
    rng = np.random.default_rng(T)
    for n in [1, 4, 5, 9, 23, 41, 72]:
        s = rand_seq(rng, n)
        bp, up, lz = emul.linear(s, 15, T)
        obp, oup = oracle.rnafold(s, 15)
        _, _, olz = oracle.fold(s)
        assert np.array_equal(bp, obp), n
        assert np.abs(up - oup).max() <= 2e-7, n
        assert abs(lz - olz) < 1e-10


@pytest.mark.parametrize("T", [64, 256])
def test_emulated_two_strand_matches_oracle(emul, oracle, T):
    rng = np.random.default_rng(100 + T)
    for n1, n2 in [(1, 1), (3, 9), (12, 9), (35, 35), (30, 52)]:
        s1, s2 = rand_seq(rng, n1), rand_seq(rng, n2)
        hp, lz = emul.cofold(s1, s2, 0.0, T)
        ohp = oracle.rnaduplex(s1, s2, 0.0)
        _, _, olz = oracle.fold(s1 + s2, n1 + 1)
        assert np.abs(hp - ohp).max() <= 2e-7, (n1, n2)
        assert abs(lz - olz) < 1e-10


def test_emulated_special_hairpins_and_dna_letters(emul, oracle):
    # BL* tetraloop list hit (GGGGAC ... src/boltzmann_param.c:5875), triloop CAACG, lower case, T
    for s in ["GGGGGACCCC", "CCAACGGG", "ggggaccuuaugc", "GGGTGACTCC", "ACAGUACUGAGCAGUACU", "NNACGUNNACGU"]:
        bp, up, lz = emul.linear(s, 5, 64)
        obp, oup = oracle.rnafold(s, 5)
        assert np.array_equal(bp, obp), s
        assert np.abs(up - oup).max() <= 2e-7, s


def test_emulated_bundled_pair(emul, oracle, bundled):
    s1, s2 = bundled["sequences"]["DIS"], bundled["sequences"]["DIS"]
    hp, _ = emul.cofold(s1, s2, 0.1, 128)
    assert np.array_equal(hp, oracle.rnaduplex(s1, s2, 0.1))


# ---- shared-memory band kernel (mcc_band.h): dense register-tiled interior sums, ring of 32 diagonals
@pytest.mark.parametrize("T", [64, 256, 512])
def test_emulated_band_linear_matches_oracle(emul, oracle, T):
    rng = np.random.default_rng(7 + T)
    for n in [1, 4, 5, 9, 23, 41, 72, 97]:
        s = rand_seq(rng, n)
        bp, up, lz = emul.linear(s, 15, T, band=True)
        obp, oup = oracle.rnafold(s, 15)
        _, _, olz = oracle.fold(s)
        assert np.abs(bp - obp).max() <= 2e-7, n
        assert np.abs(up - oup).max() <= 2e-7, n
        assert abs(lz - olz) < 1e-10


@pytest.mark.parametrize("T", [64, 256])
def test_emulated_band_two_strand_matches_oracle(emul, oracle, T):
    rng = np.random.default_rng(300 + T)
    for n1, n2 in [(1, 1), (3, 9), (12, 9), (35, 35), (30, 52), (9, 70), (61, 8)]:
        s1, s2 = rand_seq(rng, n1), rand_seq(rng, n2)
        hp, lz = emul.cofold(s1, s2, 0.0, T, band=True)
        ohp = oracle.rnaduplex(s1, s2, 0.0)
        _, _, olz = oracle.fold(s1 + s2, n1 + 1)
        assert np.abs(hp - ohp).max() <= 2e-7, (n1, n2)
        assert abs(lz - olz) < 1e-10


def test_emulated_band_special_hairpins_and_bundled(emul, oracle, bundled):
    for s in ["GGGGGACCCC", "CCAACGGG", "ggggaccuuaugc", "GGGTGACTCC", "ACAGUACUGAGCAGUACU", "NNACGUNNACGU"]:
        bp, up, lz = emul.linear(s, 5, 64, band=True)
        obp, oup = oracle.rnafold(s, 5)
        assert np.abs(bp - obp).max() <= 2e-7, s
        assert np.abs(up - oup).max() <= 2e-7, s
    s1, s2 = bundled["sequences"]["DIS"], bundled["sequences"]["DIS"]
    hp, _ = emul.cofold(s1, s2, 0.1, 128, band=True)
    assert np.array_equal(hp, oracle.rnaduplex(s1, s2, 0.1))


@pytest.mark.parametrize("W", [5, 8, 10, 15])
def test_emulated_wide_bands_match_oracle(emul, oracle, W):
    """General schedule with W-diagonal split-sum bands (far pass + near terms at the finish, long problems)."""
    rng = np.random.default_rng(7000 + W)
    for n, T in [(1, 64), (5, 64), (9, 33), (16, 64), (23, 64), (41, 32), (58, 64), (72, 256)]:
        s = rand_seq(rng, n)
        bp, up, lz = emul.linear(s, 15, T, wide=W)
        obp, oup = oracle.rnafold(s, 15)
        _, _, olz = oracle.fold(s)
        assert np.array_equal(bp, obp), n
        assert np.abs(up - oup).max() <= 2e-7, n
        assert abs(lz - olz) < 1e-10
    for n1, n2, T in [(1, 1, 64), (3, 9, 64), (12, 9, 33), (35, 35, 64), (30, 52, 128)]:
        s1, s2 = rand_seq(rng, n1), rand_seq(rng, n2)
        hp, lz = emul.cofold(s1, s2, 0.0, T, wide=W)
        ohp = oracle.rnaduplex(s1, s2, 0.0)
        _, _, olz = oracle.fold(s1 + s2, n1 + 1)
        assert np.abs(hp - ohp).max() <= 2e-7, (n1, n2)
        assert abs(lz - olz) < 1e-10


@pytest.mark.parametrize("G", [8, 16])
@pytest.mark.parametrize("T", [32, 64])
def test_emulated_cluster_matches_oracle(emul, oracle, model, G, T):
    """The wide schedule (W = 10) on a cluster of G CTAs: every rank's chunks of a diagonal dealt as on the device."""
    em = C.CDLL(str(Path(__file__).resolve().parent / "emul" / "libemul.so"))   # built by the emul fixture
    em.emul_cluster_problem.argtypes = [C.c_int, C.c_void_p, C.c_char_p] + [C.c_int] * 6 + [C.c_float, C.c_int] \
        + [C.c_void_p] * 4
    em.emul_cluster_problem.restype = C.c_int
    rng = np.random.default_rng(9000 + G + T)
    for n in [1, 5, 9, 16, 23, 41, 58, 72]:
        s = rand_seq(rng, n)
        bp = np.zeros((n + 1) * (n + 2) // 2, dtype=np.float32)
        up = np.zeros((n, 15), dtype=np.float32)
        lz = C.c_double()
        assert em.emul_cluster_problem(G, C.addressof(model), s.encode(), n, 0, 0, 15, 0, 0, 0.0, T, bp.ctypes.data,
                                       up.ctypes.data, None, C.byref(lz)) == 0
        obp, oup = oracle.rnafold(s, 15)
        _, _, olz = oracle.fold(s)
        assert np.array_equal(bp, obp), n
        assert np.abs(up - oup).max() <= 2e-7, n
        assert abs(lz.value - olz) < 1e-10
    for n1, n2 in [(1, 1), (3, 9), (12, 9), (35, 35), (30, 52)]:
        s1, s2 = rand_seq(rng, n1), rand_seq(rng, n2)
        hp = np.zeros((n1 + 1, n2 + 1), dtype=np.float32)
        lz = C.c_double()
        assert em.emul_cluster_problem(G, C.addressof(model), (s1 + s2).encode(), n1 + n2, n1 + 1, 1, 0, n1, n2, 0.0, T,
                                       None, None, hp.ctypes.data, C.byref(lz)) == 0
        ohp = oracle.rnaduplex(s1, s2, 0.0)
        _, _, olz = oracle.fold(s1 + s2, n1 + 1)
        assert np.abs(hp - ohp).max() <= 2e-7, (n1, n2)
        assert abs(lz.value - olz) < 1e-10


# ---- the device's warp-shuffle forms of the split sums, run warp by warp in lockstep (tests/emul/warp_emul.h)
TURN = 3
BAND = TURN + 2


def split_calls(n, W, T, G):
    """(side, d, i0, C) of every split-sum call of a problem of length n, as mcc_driver.h deals the rows: bands of W
    diagonals, chunks of at most wide_chunk<W>(T) rows, a problem's rows spread over G CTAs"""
    cap = (32 - (W - 1)) * (T // 32)

    def deal(first, end):
        ch = max(1, min(-(-(end - first) // G), cap))
        return [(i0, min(ch, end - i0)) for i0 in range(first, end, ch)]
    calls = []
    for d in range(TURN + 1, n):
        if (d - TURN - 1) % W == 0:
            calls += [("in", d, i0, c) for i0, c in deal(1, n - d + 1)]
    for d in range(n - 1, TURN, -1):
        if (n - 1 - d) % W == 0:
            calls += [("out", d, i0, c) for i0, c in deal(0, n - d + W - 1)]
    return calls


def edge_classes(n, W, T, G):
    """which edges of the shuffle forms' warp split the chunks of a problem reach: a warp owns 32-(W-1) rows, and a
    chunk of C rows takes NW = ceil(C/HW) warps per slice in S = (T/32)/NW slices"""
    hw = 32 - (W - 1)
    out = set()
    for _, _, _, c in split_calls(n, W, T, G):
        if c % hw in (0, 1, hw - 1):
            out.add("C%%%d=%d" % (hw, c % hw))
        nw = -(-c // hw)
        s = max(1, (T // 32) // nw)
        if nw == 1 and s > 1:
            out.add("one warp per slice")
        if s == 1:
            out.add("one slice")
    return out


@pytest.fixture(scope="module")
def lockstep(emul, model):
    em = C.CDLL(str(Path(__file__).resolve().parent / "emul" / "libemul.so"))   # built by the emul fixture
    em.emul_lockstep_problem.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_char_p] + [C.c_int] * 6 \
        + [C.c_float, C.c_int] + [C.c_void_p] * 4
    em.emul_lockstep_problem.restype = C.c_int
    em.emul_split_sums.argtypes = [C.c_void_p] + [C.c_int] * 4 + [C.c_char_p] + [C.c_int] * 4 + [C.c_uint] \
        + [C.c_void_p] * 3
    em.emul_split_sums.restype = C.c_int
    em.emul_slot_doubles.argtypes = [C.c_int]
    em.emul_slot_doubles.restype = C.c_longlong
    em.emul_outside_read_mask.argtypes = [C.c_int] * 4 + [C.c_void_p]

    class Lockstep:
        @staticmethod
        def linear(route, G, s, w, T):
            n = len(s)
            bp = np.zeros((n + 1) * (n + 2) // 2, dtype=np.float32)
            up = np.zeros((n, w), dtype=np.float32)
            lz = C.c_double()
            rc = em.emul_lockstep_problem(route, G, C.addressof(model), s.encode(), n, 0, 0, w, 0, 0, 0.0, T,
                                          bp.ctypes.data, up.ctypes.data, None, C.byref(lz))
            return rc, bp, up, lz.value

        @staticmethod
        def cofold(route, G, s1, s2, T):
            n1, n2 = len(s1), len(s2)
            hp = np.zeros((n1 + 1, n2 + 1), dtype=np.float32)
            lz = C.c_double()
            rc = em.emul_lockstep_problem(route, G, C.addressof(model), (s1 + s2).encode(), n1 + n2, n1 + 1, 1, 0,
                                          n1, n2, 0.0, T, None, None, hp.ctypes.data, C.byref(lz))
            return rc, hp, lz.value

        @staticmethod
        def split_sums(W, NB, G, T, s, cp, d, side, seed):
            n = len(s)
            bufs = [np.empty(em.emul_slot_doubles(n), dtype=np.float64) for _ in range(3)]
            rc = em.emul_split_sums(C.addressof(model), W, NB, G, T, s.encode(), n, cp, d, side, seed,
                                    *(b.ctypes.data for b in bufs))
            return (rc,) + tuple(bufs)

        @staticmethod
        def outside_read_mask(n, cp, d0, W):
            mask = np.empty(em.emul_slot_doubles(n), dtype=np.uint8)
            em.emul_outside_read_mask(n, cp, d0, W, mask.ctypes.data)
            return mask.astype(bool)

    return Lockstep()


# device configurations: (route of emul_lockstep_problem, CTAs per problem, split-sum band width)
LOCKSTEP_ROUTES = {
    "band": (1, 1, BAND),        # mcc_band_kernel: solve_band, kBatch 4
    "mcc": (0, 1, BAND),         # mcc_persistent<2,5>: solve_mcc, kBatch 2
    "wide": (10, 1, 10),         # mcc_persistent<1,10>: solve_mcc_wide<10>
    "cluster8": (10, 8, 10),     # mcc_cluster_kernel<10,8>
    "cluster16": (10, 16, 10),   # mcc_cluster_kernel<10,16>
}
# (route, T, single-strand lengths, strand-1 lengths of two-strand problems).  The long lengths put the chunk size C of
# some split-sum call on each edge class of the warp split (edge_classes; checked below); n = 1..8 are the problems
# too short for a band; strand 1 of n1 nt puts the nick cp = n1+1 just before, on and just after row 1 + 32-(W-1) (the
# second warp's first row) and, at T = 64, row 1 + 2*(32-(W-1)) (the second chunk's first row).  The clusters deal a
# chunk of ceil(rows/G): C reaches 32-(W-1)-1 = 22 rows only from n = 22*G on (175 nt for G = 8; for G = 16 the
# 355 nt this takes are left to the GPU sweep in test_gpu_parity.py).
SHORT = list(range(1, 9))
LOCKSTEP_CASES = [
    ("band", 64, [60], [27, 28, 29, 55, 56, 57]),
    ("band", 128, [60], []),
    ("band", 256, SHORT + [115], [27, 28, 29]),
    ("band", 512, [60], []),
    ("mcc", 64, [60], [55, 56, 57]),
    ("mcc", 512, SHORT + [60], [27, 28, 29]),
    ("wide", 64, [66], [22, 23, 24, 45, 46, 47]),
    ("wide", 512, SHORT + [96], [22, 23, 24]),
    ("cluster8", 32, SHORT + [175], [22, 23, 24]),
    ("cluster16", 32, SHORT + [41], [22, 23]),
]


@pytest.mark.parametrize("route,T,lengths,nicks", LOCKSTEP_CASES, ids=["%s-T%d" % (c[0], c[1]) for c in LOCKSTEP_CASES])
def test_lockstep_routes_match_oracle(lockstep, oracle, route, T, lengths, nicks):
    """Whole problems through the shuffle forms of the split sums, in the device's shared-memory sizes, against the
    oracle; every warp must meet in lockstep at every shuffle (return code 0)."""
    rid, G, W = LOCKSTEP_ROUTES[route]
    if G == 1:
        want = {"C%%%d=%d" % (32 - (W - 1), r) for r in (0, 1, 32 - W)}
        if T <= 256:   # (at T = 512 one slice takes C > 8*(32-(W-1)) rows: n > 228)
            want |= {"one warp per slice", "one slice"}
        got = set().union(*(edge_classes(n, W, T, G) for n in lengths))
        assert want <= got, sorted(want - got)
    rng = np.random.default_rng(11000 + 7 * rid + G + T)
    for n in lengths:
        s = rand_seq(rng, n)
        obp, oup = oracle.rnafold(s, 15)
        _, _, olz = oracle.fold(s)
        for w in ([15, 1] if n == max(lengths) else [15]):   # max_w = 1: PR feeds a one-nt unpaired window
            rc, bp, up, lz = lockstep.linear(rid, G, s, w, T)
            assert rc == 0, (n, w, rc)
            assert np.abs(bp - obp).max() <= 2e-7, n
            assert np.abs(up - (oup if w == 15 else oracle.rnafold(s, 1)[1])).max() <= 2e-7, (n, w)
            assert abs(lz - olz) < 1e-10, n
    for n1 in nicks:
        s1, s2 = rand_seq(rng, n1), rand_seq(rng, 24)
        rc, hp, lz = lockstep.cofold(rid, G, s1, s2, T)
        assert rc == 0, (n1, rc)
        ohp = oracle.rnaduplex(s1, s2, 0.0)
        _, _, olz = oracle.fold(s1 + s2, n1 + 1)
        assert np.abs(hp - ohp).max() <= 2e-7, n1
        assert abs(lz - olz) < 1e-10, n1


@pytest.mark.parametrize("G", [1, 8])
@pytest.mark.parametrize("T", [64, 256, 512])
@pytest.mark.parametrize("W,NB", [(BAND, 2), (BAND, 4), (10, 4)])   # kBatch: load-batch depth of the BAND forms only
def test_lockstep_split_sums_match_direct_forms(lockstep, W, NB, T, G):
    """The shuffle form against the direct form of every split-sum band on dense random tables: only the order of the
    additions differs, so both write the same cells and every element agrees to 1e-12 -- except, for two strands, the
    outside PRB / MLB cells that do not join the strands, which the outside pass never reads and the shuffle forms
    skip.  (On a real sequence most cells cannot pair and hold 0, so a shuffle that reads the wrong lane or step often
    reads one 0 for another.)"""
    rng = np.random.default_rng(12000 + W + NB + T + G)
    for n in [29, 57, 100, 130]:
        s = rand_seq(rng, n)
        starts = [("in", d) for d in range(TURN + 1, n) if (d - TURN - 1) % W == 0] \
            + [("out", d) for d in range(n - 1, TURN, -1) if (n - 1 - d) % W == 0]
        for cp in [0, n // 2 + 1]:
            for side, d in starts:
                rc, init, lock, serial = lockstep.split_sums(W, NB, G, T, s, cp, d, side == "out",
                                                             int(rng.integers(1 << 31)))
                where = (n, cp, side, d)
                assert rc == 0, where + (rc,)
                wrote = serial != init
                assert wrote.any(), where
                assert np.array_equal(lock != init, wrote), where
                read = lockstep.outside_read_mask(n, cp, d, W) if side == "out" else slice(None)
                assert np.allclose(lock[read], serial[read], rtol=1e-12, atol=0), where
