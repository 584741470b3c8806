"""SHAPE data as stacking pseudo-energies: every stack of a problem is weighted by its four bases' factors.

The soft oracle (tests/cpp/oracle_soft.c) is pinned by exhaustive enumeration that finds the stacks of each structure
itself.  CPU: the oracle, the Deigan conversion, the host planning and routing, the general kernel's routes in the host
emulator, the reactivity file reader and the command line's input errors.  GPU: the library against the soft oracle,
and byte identity wherever the data must change nothing."""
import ctypes as C
import math
import re
import subprocess
import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

from ractip_b200._lib import RpConstraint, RpOpts, RpPair, RpStackEnergy

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(Path(__file__).resolve().parent))
from conftest import rand_seq  # noqa: E402
from test_constraints import _bp_matrix, allowed_matrix, problem_view, random_constraint  # noqa: E402

TOL = 2e-7
RP_ERR_ARG = 1
CON_KEYS, CON_STACK = 1, 2
KT = (37.0 + 273.15) * 1.98717   # cal/mol
gpu = pytest.mark.gpu


def dcal(e):
    """kcal/mol -> integer 0.01 kcal/mol, half away from zero (the library's rounding)"""
    e = np.asarray(e, dtype=np.float64)
    return (np.sign(e) * np.floor(np.abs(e) * 100.0 + 0.5)).astype(np.int64)


def random_energies(rng, n):
    """integer pseudo-energies (0.01 kcal/mol): many zeros, negatives, a few large ones"""
    E = rng.integers(-300, 300, size=n)
    E[rng.random(n) < 0.3] = 0
    big = rng.random(n) < 0.08
    E[big] = rng.choice([-900, 1500, 4000], size=int(big.sum()))
    return E.astype(np.int32)


def random_reactivities(rng, n):
    r = rng.gamma(0.6, 0.8, size=n)
    r[rng.random(n) < 0.15] = -999.0   # missing
    return r


# ------------------------------------------------------------------------------------------------ soft oracle
class SoftOracle:
    def __init__(self, so, model):
        self.lib = C.CDLL(str(so))
        vp, i = C.c_void_p, C.c_int
        self.lib.orc_params_new.restype = vp
        self.lib.orc_params_new.argtypes = [vp]
        self.lib.orc_set_maxloop.argtypes = [vp, i]
        for f in (self.lib.orc_fold_soft, self.lib.orc_enumerate_soft):
            f.restype = i
            f.argtypes = [vp, C.c_char_p, i, i, vp, vp, vp, vp, i, vp]
        self.lib.orc_fold_masked.restype = i
        self.lib.orc_fold_masked.argtypes = [vp, C.c_char_p, i, i, vp, vp, vp, i, vp]
        self.lib.orc_fold.restype = i
        self.lib.orc_fold.argtypes = [vp, C.c_char_p, i, i, vp, vp, i, vp]
        self._model = model
        self.P = self.lib.orc_params_new(C.addressof(model))

    def maxloop(self, m):
        self.lib.orc_set_maxloop(self.P, m)

    @staticmethod
    def _out(n, max_w):
        return np.zeros((n + 1, n + 1)), np.zeros((n, max(max_w, 1))), C.c_double()

    def _call(self, f, seq, cp, allow, E, max_w):
        n = len(seq)
        pr, up, lz = self._out(n, max_w)
        a = None if allow is None else np.ascontiguousarray(allow, dtype=np.uint8)
        e = None if E is None else np.ascontiguousarray(E, dtype=np.int32)
        assert e is None or e.shape == (n,)
        rc = f(self.P, seq.encode(), n, cp, None if a is None else a.ctypes.data, None if e is None else e.ctypes.data,
               pr.ctypes.data, up.ctypes.data, max_w, C.byref(lz))
        assert rc == 0
        return pr, (up if max_w > 0 else None), lz.value

    def fold(self, seq, cp=0, allow=None, E=None, max_w=0):
        return self._call(self.lib.orc_fold_soft, seq, cp, allow, E, max_w)

    def enumerate(self, seq, cp=0, allow=None, E=None, max_w=0):
        return self._call(self.lib.orc_enumerate_soft, seq, cp, allow, E, max_w)

    def fold_masked(self, seq, cp, allow, max_w):
        n = len(seq)
        pr, up, lz = self._out(n, max_w)
        a = np.ascontiguousarray(allow, dtype=np.uint8)
        assert self.lib.orc_fold_masked(self.P, seq.encode(), n, cp, a.ctypes.data, pr.ctypes.data, up.ctypes.data,
                                        max_w, C.byref(lz)) == 0
        return pr, up, lz.value

    def fold_plain(self, seq, cp, max_w):
        n = len(seq)
        pr, up, lz = self._out(n, max_w)
        assert self.lib.orc_fold(self.P, seq.encode(), n, cp, pr.ctypes.data, up.ctypes.data, max_w, C.byref(lz)) == 0
        return pr, up, lz.value


def _cc(cmd):
    subprocess.run(cmd, check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)


@pytest.fixture(scope="module")
def sorc(tmp_path_factory, model):
    so = tmp_path_factory.mktemp("sorc") / "liboracle_soft.so"
    _cc(["gcc", "-O3", "-fPIC", "-shared", "-I", str(ROOT / "include"), str(ROOT / "tests" / "cpp" / "oracle_soft.c"),
         "-o", str(so), "-lm"])
    o = SoftOracle(so, model)
    yield o
    o.maxloop(30)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = tmp_path_factory.mktemp("sshim") / "libshape_shim.so"
    csrc = ROOT / "ractip_b200" / "csrc"
    _cc(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", str(ROOT / "include"), "-I", str(csrc),
         str(csrc / "plan.cpp"), str(ROOT / "tests" / "cpp" / "shape_shim.cpp"), "-o", str(so)])
    lib = C.CDLL(str(so))
    vp = C.c_void_p
    lib.shape_shim.argtypes = [vp, vp, vp, C.c_int, vp, C.c_char_p, C.c_int, vp, vp, C.c_int, vp, vp]
    lib.shape_shim.restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def kemul(tmp_path_factory):
    so = tmp_path_factory.mktemp("semul") / "libemul_shaped.so"
    d = ROOT / "tests" / "emul"
    _cc(["g++", "-O2", "-U_FORTIFY_SOURCE", "-std=c++17", "-fPIC", "-shared", "-I", str(ROOT / "ractip_b200" / "csrc"),
         "-I", str(ROOT / "include"), "-o", str(so), str(d / "emul_shaped.cpp"),
         str(ROOT / "ractip_b200" / "csrc" / "dev_model.cpp")])
    lib = C.CDLL(str(so))
    vp, i = C.c_void_p, C.c_int
    lib.emul_shaped_problem.argtypes = [i, i, i, vp, vp, vp, C.c_char_p, i, i, i, i, i, i, C.c_float, i, vp, vp, vp, vp]
    lib.emul_shaped_problem.restype = i
    return lib


def opts(**kw):
    o = dict(max_w=15, min_w=5, th_ss=0.5, th_hy=0.1, th_ac=0.003, use_pf_duplex=0)
    o.update(kw)
    return RpOpts(**o)


# ------------------------------------------------------------------------ soft oracle vs enumeration (CPU)
def _check_enum(sorc, seq, cp, allow, E, max_w):
    pr, up, lz = sorc.fold(seq, cp, allow, E, max_w)
    epr, eup, elz = sorc.enumerate(seq, cp, allow, E, max_w)
    assert abs(lz - elz) < 1e-12 * max(1.0, abs(elz))
    np.testing.assert_allclose(pr, epr, rtol=0, atol=1e-12)
    if max_w:
        np.testing.assert_allclose(up, eup, rtol=0, atol=1e-12)
    return lz


@pytest.mark.parametrize("maxloop", [30, 3])
def test_soft_oracle_single_strand(sorc, maxloop):
    sorc.maxloop(maxloop)
    try:
        rng = np.random.default_rng(51)
        moved = 0
        for k in range(8):
            n = int(rng.integers(12, 19))
            s = rand_seq(rng, n) if k else "GGGGAAACCCCAGGGAAAC"[:n]
            E = random_energies(rng, n)
            allow = None
            if k % 2:
                m, bp, unp = problem_view(random_constraint(rng, n, 0)[0], None, n, 0, 0)
                allow = allowed_matrix(m, bp, unp)
            lz = _check_enum(sorc, s, 0, allow, E, 6)
            moved += abs(lz - sorc.fold(s, 0, allow, None, 0)[2]) > 1e-6
        assert moved >= 4   # the energies do change the ensembles
    finally:
        sorc.maxloop(30)


@pytest.mark.parametrize("maxloop", [30, 3])
def test_soft_oracle_two_strands(sorc, maxloop):
    sorc.maxloop(maxloop)
    try:
        rng = np.random.default_rng(52)
        cases = [("GGGAAUCC", "GGAUUCCC"), ("GCGCAAAG", "CUUUGCGC")]
        for _ in range(5):
            n1, n2 = int(rng.integers(6, 10)), int(rng.integers(6, 9))
            cases.append((rand_seq(rng, n1), rand_seq(rng, n2)))
        for k, (s1, s2) in enumerate(cases):
            n1, n2 = len(s1), len(s2)
            E = random_energies(rng, n1 + n2)
            allow = None
            if k % 2:
                m, bp, unp = problem_view(*random_constraint(rng, n1, n2), n1, n2, 2)
                allow = allowed_matrix(m, bp, unp)
            _check_enum(sorc, s1 + s2, n1 + 1, allow, E, 0)
    finally:
        sorc.maxloop(30)


def test_soft_oracle_intermolecular_stacks_carry_nothing(sorc):
    """Energies on the bases of a co-fold's intermolecular helix only: the ensemble of pure duplexes is unchanged."""
    s1, s2 = "GGGG", "CCCC"   # too short to fold alone: every structure is intermolecular
    E = np.array([-500, 700, 300, -200, 900, -400, 250, 100], dtype=np.int32)
    pr, _, lz = sorc.fold(s1 + s2, 5, None, E, 0)
    pr0, _, lz0 = sorc.fold(s1 + s2, 5, None, None, 0)
    assert lz == lz0 and np.array_equal(pr, pr0)
    _check_enum(sorc, s1 + s2, 5, None, E, 0)


def test_soft_oracle_zero_energies_are_bitwise_the_oracle(sorc):
    rng = np.random.default_rng(53)
    for n, cp in ((40, 0), (30, 17)):
        s = rand_seq(rng, n)
        w = 8 if cp == 0 else 0
        zero = np.zeros(n, dtype=np.int32)
        for E in (None, zero):
            a = sorc.fold(s, cp, None, E, w)
            b = sorc.fold_plain(s, cp, w)
            assert a[2] == b[2] and np.array_equal(a[0], b[0]) and (w == 0 or np.array_equal(a[1], b[1]))
        n1 = cp - 1 if cp else n
        m, bp, unp = problem_view(*random_constraint(rng, n1, n - n1), n1, n - n1, 2 if cp else 0)
        allow = allowed_matrix(m, bp, unp)
        a = sorc.fold(s, cp, allow, zero, w)
        b = sorc.fold_masked(s, cp, allow, w)
        assert a[2] == b[2] and np.array_equal(a[0], b[0]) and (w == 0 or np.array_equal(a[1], b[1]))


# ----------------------------------------------------------------------------------------- Deigan (CPU)
def test_shape_deigan(lib):
    from ractip_b200 import shape_deigan
    r = np.array([-999.0, -0.5, np.nan, 0.0, math.e - 1, 1.0, 3.0])
    e = shape_deigan(r)
    want = [0.0, 0.0, 0.0, -0.6, 1.8 - 0.6, 1.8 * math.log(2) - 0.6, 1.8 * math.log(4) - 0.6]
    np.testing.assert_allclose(e, want, rtol=0, atol=1e-15)
    assert e[0] == 0 and e[2] == 0 and e[3] == -0.6
    np.testing.assert_allclose(shape_deigan(r, 2.6, -0.8)[3:], 2.6 * np.log(r[3:] + 1) - 0.8, rtol=0, atol=1e-15)
    assert shape_deigan([]).shape == (0,)
    assert lib.rp_shape_deigan(None, 3, 1.8, -0.6, None) == RP_ERR_ARG


# --------------------------------------------------------------------------------------- planning (CPU)
def plan(shim, pairs, energies, cons=None, o=None):
    """(rc, message, factor buffer, per-problem (seq_off, n, constrained, general), same plan as without energies)"""
    keep = []
    arr = (RpPair * len(pairs))()
    sarr = (RpStackEnergy * len(pairs))()
    carr = (RpConstraint * len(pairs))() if cons else None
    for k, (s1, s2) in enumerate(pairs):
        b = [s1.encode(), s2.encode()]
        keep.append(b)
        arr[k].s1, arr[k].n1, arr[k].s2, arr[k].n2 = b[0], len(s1), b[1] or None, len(s2)
        for s, e in enumerate(energies[k] if energies[k] is not None else (None, None)):
            if e is not None:
                a = np.ascontiguousarray(e, dtype=np.float64)
                keep.append(a)
                setattr(sarr[k], f"e{s + 1}", a.ctypes.data)
        if cons:
            c = [x.encode() if x is not None else None for x in cons[k]]
            keep.append(c)
            carr[k].c1, carr[k].c2 = c
    cap = sum(2 * (len(a) + len(b)) + 4 for a, b in pairs) + 16
    stack = np.zeros(cap)
    slen = C.c_longlong()
    probs = np.zeros((3 * len(pairs), 4), dtype=np.int64)
    msg = C.create_string_buffer(256)
    same = C.c_int()
    rc = shim.shape_shim(arr, carr, sarr, len(pairs), C.byref(o or opts()), msg, 256, stack.ctypes.data, C.byref(slen),
                         cap, probs.ctypes.data, C.byref(same))
    return rc, msg.value.decode(), stack[:slen.value], probs, bool(same.value)


def test_plan_flags_routes_and_factors(shim):
    rng = np.random.default_rng(61)
    pairs = [("ACGU" * 18, "ACGU" * 34)] * 4
    e1 = rng.normal(0, 1, 72)
    e2 = rng.normal(0, 1, 136)
    rc, msg, stack, probs, _ = plan(shim, pairs, [None, (e1, None), (None, e2), (np.zeros(72), np.zeros(136))])
    assert rc == 0, msg
    assert probs[:, 2].tolist() == [0, 0, 0, 2, 0, 2, 0, 2, 2, 0, 0, 0]
    assert probs[:, 3].tolist() == [0, 0, 0, 1, 0, 1, 0, 1, 1, 0, 0, 0]   # band kernel without data
    f1, f2 = np.exp(-dcal(e1) * 10.0 / KT), np.exp(-dcal(e2) * 10.0 / KT)
    off = {k: int(probs[k, 0]) for k in range(12)}
    close = lambda a, b: np.testing.assert_allclose(a, b, rtol=1e-15, atol=0)   # libm's exp against numpy's
    close(stack[off[3]:off[3] + 72], f1)
    close(stack[off[5]:off[5] + 208], np.concatenate([f1, np.ones(136)]))
    close(stack[off[7]:off[7] + 136], f2)
    close(stack[off[8]:off[8] + 208], np.concatenate([np.ones(72), f2]))
    assert np.array_equal(stack[off[3]:off[3] + 72], stack[off[5]:off[5] + 72])
    others = np.ones(len(stack), dtype=bool)
    for k, m in ((3, 72), (5, 208), (7, 136), (8, 208)):
        others[off[k]:off[k] + m] = False
    assert np.all(stack[others] == 1.0)
    # with -c keys on the same pair: both bits, and the constrained problems stay on the general kernel
    cons = [(None, None), ("(" + "." * 70 + ")", None), (None, None), (None, None)]
    rc, msg, _, probs, _ = plan(shim, pairs, [None, (e1, None), None, None], cons)
    assert rc == 0, msg
    assert probs[3:6, 2].tolist() == [CON_KEYS | CON_STACK, 0, CON_KEYS | CON_STACK]
    # --duplex: the hybridization takes no pseudo-energies
    rc, _, _, probs, _ = plan(shim, pairs, [None, (e1, None), None, None], o=opts(use_pf_duplex=1))
    assert rc == 0 and probs[3, 2] == CON_STACK and probs[5, 2] == 0 and probs[5, 3] == 1   # duplex_kernel's queue


def test_plan_without_data_is_the_plain_plan(shim):
    pairs = [("ACGU" * 18, "ACGU" * 34), ("GGGAAACCC" * 3, "")]
    for energies in ([None, None], [(None, None), (None, None)],
                     [(np.zeros(72), np.zeros(136)), (np.full(27, 0.0049), None)],
                     [(np.full(72, -0.00499), None), (np.zeros(27), None)]):
        rc, msg, stack, probs, same = plan(shim, pairs, energies)
        assert rc == 0, msg
        assert len(stack) == 0 and same and not probs[:, 2].any()


def test_plan_rounding_boundary(shim):
    pairs = [("GGGAAACCC", "")]
    e = np.array([0.005, -0.005, 0.0049999, -0.0049999, 0.015, -0.025, 1.234, 0.0, 0.0])
    rc, msg, stack, probs, same = plan(shim, pairs, [(e, None)])
    assert rc == 0 and probs[0, 2] == CON_STACK and not same
    want = np.exp(-np.array([1, -1, 0, 0, 2, -3, 123, 0, 0]) * 10.0 / KT)
    off = int(probs[0, 0])
    np.testing.assert_allclose(stack[off:off + 9], want, rtol=1e-15, atol=0)
    assert np.count_nonzero(stack[off:off + 9] == 1.0) == 4
    np.testing.assert_array_equal(dcal(e), [1, -1, 0, 0, 2, -3, 123, 0, 0])


@pytest.mark.parametrize("bad,where", [
    (float("nan"), "pair 1, e2, position 3: nan kcal/mol is not finite"),
    (float("inf"), "pair 1, e2, position 3: inf kcal/mol is not finite"),
    (float("-inf"), "pair 1, e2, position 3: -inf kcal/mol is not finite")])
def test_non_finite_energies(shim, bad, where):
    e2 = np.zeros(4)
    e2[2] = bad
    rc, msg, _, _, _ = plan(shim, [("ACGU" * 5, "ACGU"), ("GGGAAACCC", "GGGU")], [(np.ones(20), None), (None, e2)])
    assert rc == RP_ERR_ARG and msg == where


# ------------------------------------------------------------------------------------------ emulator (CPU)
ROUTES = [(0, 1), (5, 1), (10, 1), (15, 1), (10, 8), (10, 16)]


def _emul(kemul, model, f, seq, cp, kind, max_w, n1, n2, route, G, lockstep, T=64):
    n = len(seq)
    bp = np.zeros((n + 1) * (n + 2) // 2, dtype=np.float32)
    up = np.zeros((n, max(max_w, 1)), dtype=np.float32)
    hp = np.zeros((n1 + 1, n2 + 1), dtype=np.float32)
    lz = C.c_double()
    stk = np.ascontiguousarray(np.concatenate([[1.0], f]))   # stk[1..n]
    rc = kemul.emul_shaped_problem(route, G, int(lockstep), stk.ctypes.data, None, C.addressof(model), seq.encode(), n,
                                   cp, kind, max_w, n1, n2, 0.1, T, bp.ctypes.data, up.ctypes.data, hp.ctypes.data,
                                   C.byref(lz))
    assert rc == 0, rc
    return bp, up, hp, lz.value


@pytest.mark.parametrize("lockstep", [False, True])
def test_emulator_routes(kemul, sorc, model, lockstep):
    rng = np.random.default_rng(71)
    s1, s2 = rand_seq(rng, 47), rand_seq(rng, 38)
    E1, E2 = random_energies(rng, 47), random_energies(rng, 38)
    f1, f2 = np.exp(-E1 * 10.0 / KT), np.exp(-E2 * 10.0 / KT)
    pr1, up1, lz1 = sorc.fold(s1, 0, None, E1, 8)
    pr12, _, lz12 = sorc.fold(s1 + s2, 48, None, np.concatenate([E1, E2]), 0)
    want = np.zeros((48, 39))
    want[1:, 1:] = pr12[1:48, 48:]
    want = np.where((want >= 0.1) & (want.astype(np.float32) > np.float32(0.1)), want, 0)
    for route, G in ROUTES:
        b, u, _, lz = _emul(kemul, model, f1, s1, 0, 0, 8, 47, 0, route, G, lockstep)
        np.testing.assert_allclose(_bp_matrix(b, 47), pr1, rtol=0, atol=TOL)
        np.testing.assert_allclose(u, up1, rtol=0, atol=TOL)
        assert abs(lz - lz1) < 1e-10, (route, G)
        _, _, h, lz = _emul(kemul, model, np.concatenate([f1, f2]), s1 + s2, 48, 1, 0, 47, 38, route, G, lockstep)
        np.testing.assert_allclose(h, want, rtol=0, atol=TOL)
        assert abs(lz - lz12) < 1e-10, (route, G)


# ------------------------------------------------------------------------------------------ front end (CPU)
def test_read_shape(tmp_path, lib):
    from ractip_b200.frontend import read_shape
    p = tmp_path / "r.shape"
    p.write_text("# probing\n1 G 0.5\n\n3 g 1.25\n4 -999\n6 T 0.0\n")
    r = read_shape(str(p), "GGGAAU")
    assert r[0] == 0.5 and r[2] == 1.25 and r[3] == -999 and r[5] == 0.0
    assert np.isnan(r[1]) and np.isnan(r[4])
    for text, msg in (("7 U 0.5\n", "line 1: position 7 is outside 1..6"),
                      ("0 0.5\n", "position 0 is outside"),
                      ("2 0.5\n2 0.7\n", "line 2: position 2 is listed twice"),
                      ("1 A 0.5\n", "nucleotide 'A' at position 1, the sequence has 'G'"),
                      ("1 G x\n", "value 'x' is not a number"),
                      ("1 G inf\n", "value 'inf' is not finite"),
                      ("a G 1\n", "position 'a' is not an integer"),
                      ("1 G 0.5 7\n", "expected 'position [nucleotide] value'")):
        p.write_text(text)
        with pytest.raises(ValueError, match=re.escape(msg)):
            read_shape(str(p), "GGGAAU")


def test_predict_passes_energies_and_leaves_shuffles_bare(monkeypatch):
    from ractip_b200 import frontend, shape_deigan
    from ractip_b200.frontend import FastaRecord
    calls = []

    class Stop(Exception):
        pass

    class FakeStage:
        model = None

        def run_dense(self, seqs, opts, constraints=None, **kw):
            calls.append((list(seqs), constraints, kw))
            if len(calls) == 2:
                raise Stop
            return [SimpleNamespace(bp1=None, bp2=None) for _ in seqs]

    monkeypatch.setattr(frontend, "solve_joint", lambda *a, **k: None)
    monkeypatch.setattr(frontend, "solve_ss", lambda *a, **k: (None, None, 0.0))
    a, b = FastaRecord("a", "GGGAAACCC"), FastaRecord("b", "GGGUUUCCC")
    r = np.array([0.1, 0.2, -1, 0.4, 1.5, 0, 0, 2, 3])
    with pytest.raises(Stop):
        frontend.predict(FakeStage(), [(a, b)], zscore=12, num_shuffling=3, shape={"b": r}, shape_slope=2.0)
    (e1, e2), = calls[0][2]["stack_energies"]
    assert e1 is None and np.array_equal(e2, shape_deigan(r, 2.0, -0.6))
    assert len(calls[1][0]) == 3 and calls[1][2] == {}
    with pytest.raises(ValueError, match="reactivities for c: no such record"):
        frontend.predict(FakeStage(), [(a, b)], shape={"c": r})


def _cli(args, cwd=ROOT):
    return subprocess.run([sys.executable, "-m", "ractip_b200"] + args, cwd=cwd, stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True, timeout=600)


def test_command_line_input_errors(tmp_path, lib, bundled):
    seqs = bundled["sequences"]
    (tmp_path / "a.fa").write_text(f">MicA\n{seqs['MicA']}\n")
    (tmp_path / "b.fa").write_text(f">ompA\n{seqs['ompA']}\n")
    (tmp_path / "ok.shape").write_text("1 0.5\n")
    (tmp_path / "bad.shape").write_text(f"{len(seqs['MicA']) + 1} 0.5\n")
    fa = [str(tmp_path / "a.fa"), str(tmp_path / "b.fa")]
    for extra, msg in ((["--shape", f"SodB={tmp_path / 'ok.shape'}"], "no record named 'SodB'"),
                       (["--shape", f"MicA={tmp_path / 'bad.shape'}"], "is outside 1..72"),
                       (["--shape", f"MicA={tmp_path / 'none.shape'}"], "No such file"),
                       (["--shape", "MicA"], "expected NAME=FILE")):
        r = _cli(extra + fa)
        assert r.returncode == 1 and msg in r.stdout, r.stdout


# ------------------------------------------------------------------------------------------------- GPU
def _stage_env(monkeypatch, env):
    from ractip_b200 import ProbabilityStage
    for k in ("RP_BAND", "RP_CLUSTER", "RP_MCC_LONG_N"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    return ProbabilityStage()


def _oracle_pair(sorc, s1, s2, e1, e2, o, c1=None, c2=None):
    """the soft oracle's (pr, up, logZ) of the three problems, from kcal/mol energies as the library takes them"""
    n1, n2 = len(s1), len(s2)
    E1 = dcal(e1) if e1 is not None else np.zeros(n1, dtype=np.int64)
    E2 = dcal(e2) if e2 is not None else np.zeros(n2, dtype=np.int64)
    out = {}
    for which, seq, E in ((0, s1, E1), (1, s2, E2), (2, s1 + s2, np.concatenate([E1, E2]))):
        A = None
        if c1 is not None or c2 is not None:
            m, bp, unp = problem_view(c1, c2, n1, n2, which)
            A = allowed_matrix(m, bp, unp)
        out[which] = sorc.fold(seq, n1 + 1 if which == 2 else 0, A, E, 0 if which == 2 else o.max_w)
    return out


def _hp_want(pr, n1, n2, th):
    want = np.zeros((n1 + 1, n2 + 1))
    want[1:, 1:] = pr[1:n1 + 1, n1 + 1:]
    return np.where((want >= th) & (want.astype(np.float32) > np.float32(th)), want, 0)


def _compare(r, lz, orc, n1, n2, o):
    for which, (bp, nn, up) in ((0, (r.bp1, n1, r.up1)), (1, (r.bp2, n2, r.up2))):
        pr, oup, olz = orc[which]
        np.testing.assert_allclose(_bp_matrix(bp, nn), pr, rtol=0, atol=TOL)
        np.testing.assert_allclose(up, oup, rtol=0, atol=TOL)
        assert abs(lz[which] - olz) < 1e-9
    pr, _, olz = orc[2]
    np.testing.assert_allclose(r.hp, _hp_want(pr, n1, n2, o.th_hy), rtol=0, atol=TOL)
    assert abs(lz[2] - olz) < 1e-9


def _run(stage, pairs, o, cons=None, energies=None):
    b = stage.batch(pairs, o, cons, energies)
    try:
        b.run()
        flat = b.fetch_dense()
        return b.split_dense(flat), b.fetch_logz(), flat.copy()
    finally:
        b.close()


def _bundled_energies(bundled):
    from ractip_b200 import shape_deigan
    seqs = bundled["sequences"]
    rng = np.random.default_rng(81)
    pairs = [(seqs[a], seqs[b]) for a, b in bundled["pairs"]]
    energies = [(shape_deigan(random_reactivities(rng, len(s1))), shape_deigan(random_reactivities(rng, len(s2))))
                for s1, s2 in pairs]
    return pairs, energies


@gpu
@pytest.mark.parametrize("env", [{}, {"RP_BAND": "0"}], ids=["default", "no_band"])
def test_gpu_bundled_pairs(sorc, bundled, monkeypatch, env):
    pairs, energies = _bundled_energies(bundled)
    o = opts()
    stage = _stage_env(monkeypatch, env)
    try:
        res, lz, _ = _run(stage, pairs, o, energies=energies)
        for (s1, s2), (e1, e2), r, z in zip(pairs, energies, res, lz):
            _compare(r, z, _oracle_pair(sorc, s1, s2, e1, e2, o), len(s1), len(s2), o)
        # sparse lists and tensors of the shaped batch agree with its dense fetch
        recs = stage.run_sparse(pairs, o, stack_energies=energies)
        for (s1, s2), r, sp in zip(pairs, res, recs):
            n1, n2 = len(s1), len(s2)
            P1 = _bp_matrix(r.bp1, n1)
            want_x = sorted((i - 1, j - 1) for i in range(1, n1 + 1) for j in range(i + 1, n1 + 1) if P1[i, j] > o.th_ss)
            assert sorted((int(x["i"]), int(x["j"])) for x in sp.x) == want_x
            want_z = sorted((i - 1, j - 1) for i in range(1, n1 + 1) for j in range(1, n2 + 1) if r.hp[i, j] > o.th_hy)
            assert sorted((int(x["i"]), int(x["j"])) for x in sp.z) == want_z
        import torch
        b = stage.batch(pairs, o, None, energies)
        try:
            b.run()
            t = b.tensors()
            torch.cuda.synchronize()
            for k, r in enumerate(res):
                n1, n2 = len(pairs[k][0]), len(pairs[k][1])
                np.testing.assert_array_equal(t["hp"][k, :n1 + 1, :n2 + 1].cpu().numpy(), r.hp)
                np.testing.assert_array_equal(np.triu(t["bp1"][k, :n1 + 1, :n1 + 1].cpu().numpy(), 1),
                                              _bp_matrix(r.bp1, n1).astype(np.float32))
                np.testing.assert_array_equal(t["up2"][k, :n2].cpu().numpy(), r.up2)
        finally:
            b.close()
    finally:
        stage.close()


_LONG = {}


def _long_case(sorc):
    if not _LONG:
        from ractip_b200 import shape_deigan
        rng = np.random.default_rng(82)
        o = opts()
        pairs = [(rand_seq(rng, 620), rand_seq(rng, 300)), (rand_seq(rng, 720), rand_seq(rng, 90))]
        energies = [(shape_deigan(random_reactivities(rng, len(a))), shape_deigan(random_reactivities(rng, len(b))))
                    for a, b in pairs]
        _LONG["case"] = (pairs, energies, [_oracle_pair(sorc, a, b, e1, e2, o) for (a, b), (e1, e2) in zip(pairs, energies)])
    return _LONG["case"]


ROUTE_ENVS = [{}, {"RP_MCC_LONG_N": "1", "RP_CLUSTER": "0"}, {"RP_CLUSTER": "8"}, {"RP_CLUSTER": "16"}]


@gpu
@pytest.mark.parametrize("env", ROUTE_ENVS, ids=["default", "wide", "cluster8", "cluster16"])
def test_gpu_long_pair_routes(sorc, monkeypatch, env):
    pairs, energies, orc = _long_case(sorc)
    o = opts()
    stage = _stage_env(monkeypatch, env)
    try:
        res, lz, _ = _run(stage, pairs, o, energies=energies)
    finally:
        stage.close()
    for (s1, s2), r, z, oc in zip(pairs, res, lz, orc):
        _compare(r, z, oc, len(s1), len(s2), o)


@gpu
def test_gpu_byte_identity(bundled, monkeypatch):
    seqs, dis = bundled["sequences"], bundled["readme_dis"]
    pairs = [(seqs[a], seqs[b]) for a, b in (("MicA", "ompA"), ("DIS", "DIS"), ("OxyS", "fhlA"))]
    o = opts()
    rng = np.random.default_rng(83)
    from ractip_b200 import shape_deigan
    stage = _stage_env(monkeypatch, {})
    try:
        # all-missing reactivities: no data
        _, lz0, plain = _run(stage, pairs, o)
        missing = [(shape_deigan(np.full(len(a), -999.0)), shape_deigan(np.full(len(b), -999.0))) for a, b in pairs]
        _, lz1, flat = _run(stage, pairs, o, energies=missing)
        assert plain.tobytes() == flat.tobytes() and lz0.tobytes() == lz1.tobytes()
        # the unshaped pairs of a mixed batch against the same pairs alone
        shaped = (shape_deigan(random_reactivities(rng, len(pairs[0][0]))), None)
        r1, lz1, _ = _run(stage, pairs, o, energies=[shaped, None, (None, None)])
        r0, lz0, _ = _run(stage, pairs[1:], o)
        for k in (1, 2):
            for f in ("bp1", "bp2", "up1", "up2", "hp"):
                assert getattr(r1[k], f).tobytes() == getattr(r0[k - 1], f).tobytes()
            assert lz1[k].tobytes() == lz0[k - 1].tobytes()
        assert r1[0].bp1.tobytes() != _run(stage, pairs[:1], o)[0][0].bp1.tobytes()   # the data did reach pair 0
        # --duplex: the hybridization ignores the data
        od = opts(use_pf_duplex=1)
        d0, _, _ = _run(stage, pairs, od)
        both = [(shape_deigan(random_reactivities(rng, len(a))), shape_deigan(random_reactivities(rng, len(b))))
                for a, b in pairs]
        d1, _, _ = _run(stage, pairs, od, energies=both)
        for k in range(3):
            assert d0[k].hp.tobytes() == d1[k].hp.tobytes()
        # constrained-only batches: the same bytes through rp_batch_create_soft as through rp_batch_create_constrained
        cons = [None, (dis["s1"], dis["s2"]), None]
        _, lzc, fc = _run(stage, pairs, o, cons=cons)
        _, lzs, fs = _run(stage, pairs, o, cons=cons, energies=[None] * 3)
        _, lzz, fz = _run(stage, pairs, o, cons=cons, energies=missing)
        assert fc.tobytes() == fs.tobytes() == fz.tobytes() and lzc.tobytes() == lzs.tobytes() == lzz.tobytes()
    finally:
        stage.close()


@gpu
def test_gpu_constraints_with_shape(sorc, bundled, monkeypatch):
    from ractip_b200 import shape_deigan
    seqs, dis = bundled["sequences"], bundled["readme_dis"]
    rng = np.random.default_rng(84)
    pairs = [(seqs["DIS"], seqs["DIS"]), (seqs["MicA"], seqs["ompA"])]
    cons = [(dis["s1"], dis["s2"]), random_constraint(rng, 72, 137, dens=0.15)]
    energies = [(shape_deigan(random_reactivities(rng, len(a))), shape_deigan(random_reactivities(rng, len(b))))
                for a, b in pairs]
    o = opts()
    stage = _stage_env(monkeypatch, {})
    try:
        res, lz, _ = _run(stage, pairs, o, cons=cons, energies=energies)
    finally:
        stage.close()
    for (s1, s2), (c1, c2), (e1, e2), r, z in zip(pairs, cons, energies, res, lz):
        _compare(r, z, _oracle_pair(sorc, s1, s2, e1, e2, o, c1, c2), len(s1), len(s2), o)


def _pack_bp(pr, n):
    bp = np.zeros((n + 1) * (n + 2) // 2, dtype=np.float32)
    for i in range(1, n + 1):
        off = i * (2 * n + 1 - i) // 2
        bp[off + i + 1:off + n + 1] = pr[i, i + 1:]
    return bp


@gpu
def test_gpu_command_line(sorc, model, bundled, tmp_path):
    from ractip_b200 import bp_offsets, default_ip_opts, shape_deigan, solve_joint
    from ractip_b200.frontend import read_shape
    from ractip_b200.stage import PairProbabilities
    seqs = bundled["sequences"]
    s1, s2 = seqs["MicA"], seqs["ompA"]
    rng = np.random.default_rng(85)
    (tmp_path / "a.fa").write_text(f">MicA\n{s1}\n")
    (tmp_path / "b.fa").write_text(f">ompA\n{s2}\n")
    lines = [f"{i + 1} {s1[i]} {v:.4f}" for i, v in enumerate(random_reactivities(rng, len(s1))) if v >= 0]
    (tmp_path / "MicA.shape").write_text("\n".join(lines) + "\n")
    r = _cli(["--shape", f"MicA={tmp_path / 'MicA.shape'}", str(tmp_path / "a.fa"), str(tmp_path / "b.fa")])
    assert r.returncode == 0, r.stdout
    out = r.stdout.splitlines()
    e1 = shape_deigan(read_shape(str(tmp_path / "MicA.shape"), s1))
    o = opts()
    orc = _oracle_pair(sorc, s1, s2, e1, None, o)
    P = PairProbabilities(_pack_bp(orc[0][0], len(s1)), bp_offsets(len(s1)), orc[0][1].astype(np.float32),
                          _pack_bp(orc[1][0], len(s2)), bp_offsets(len(s2)), orc[1][1].astype(np.float32),
                          _hp_want(orc[2][0], len(s1), len(s2), o.th_hy).astype(np.float32))
    j = solve_joint(model, s1, s2, P, default_ip_opts())
    assert out[0] == ">MicA" and out[2] == j.r1 and out[5] == j.r2, (out, j.r1, j.r2)
