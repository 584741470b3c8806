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
