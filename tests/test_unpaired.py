"""Unpaired pseudo-energies (RNAfold --shapeMethod=W): every base a structure leaves unpaired is weighted by its factor.

The kernel applies them as pair factors (pair_sc, mcc_core.h); the probed oracle (tests/cpp/oracle_probed.c) applies
them literally to every unpaired base of every loop and window, and is pinned by exhaustive enumeration.  CPU: the
oracle, the host planning and its range check, the general kernel's routes in the host emulator (serial and
warp-lockstep), sampling against the exact distribution, the front end.  GPU: the library against the probed oracle,
byte identity wherever the data must change nothing, samples against the emulator, sparse lists, tensors and the
command line."""
import ctypes as C
import math
import re
import subprocess
import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

from ractip_b200._lib import RpConstraint, RpOpts, RpPair, RpStackEnergy, RpUnpairedEnergy

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(Path(__file__).resolve().parent))
from conftest import rand_seq  # noqa: E402
from test_constraints import _bp_matrix, allowed_matrix, problem_view, random_constraint  # noqa: E402
from test_ip import all_structures, can_pair, to_string  # noqa: E402

TOL = 2e-7
RP_ERR_ARG, RP_ERR_UNSUPPORTED = 1, 10
CON_KEYS, CON_STACK, CON_SAMPLE, CON_UNPAIRED = 1, 2, 4, 8
KT = (37.0 + 273.15) * 1.98717   # cal/mol
MAX_B = 150 * math.log(10)
ROUTES = [(0, 1), (5, 1), (10, 1), (15, 1), (10, 8), (10, 16)]
ROUTE_ENVS = [{}, {"RP_MCC_LONG_N": "1", "RP_CLUSTER": "0"}, {"RP_CLUSTER": "8"}, {"RP_CLUSTER": "16"}]
gpu = pytest.mark.gpu


def dcal(e):
    """kcal/mol -> integer 0.01 kcal/mol, half away from zero (the library's rounding)"""
    e = np.asarray(e, dtype=np.float64)
    return (np.sign(e) * np.floor(np.abs(e) * 100.0 + 0.5)).astype(np.int64)


def random_unpaired(rng, n, scale=150):
    """integer unpaired pseudo-energies (0.01 kcal/mol): zeros, both signs, a few large ones"""
    U = rng.integers(-scale, scale, size=n)
    U[rng.random(n) < 0.3] = 0
    big = rng.random(n) < 0.06
    U[big] = rng.choice([-400, 600], size=int(big.sum()))
    return U.astype(np.int32)


def random_kcal(rng, n, scale=0.5):
    """unpaired pseudo-energies in kcal/mol as a user brings them (a perturbation vector), B well inside the range"""
    u = rng.normal(0, scale, n)
    u[rng.random(n) < 0.2] = 0.0
    return u


def _cc(cmd):
    subprocess.run(cmd, check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)


def _ptr(a, dtype):
    if a is None:
        return None, None
    a = np.ascontiguousarray(a, dtype=dtype)
    return a, a.ctypes.data


# ---------------------------------------------------------------------------------------------- probed oracle
class ProbedOracle:
    def __init__(self, so, model):
        self.lib = C.CDLL(str(so))
        vp, i = C.c_void_p, C.c_int
        self.lib.orc_params_new.restype = vp
        self.lib.orc_params_new.argtypes = [vp]
        self.lib.orc_set_maxloop.argtypes = [vp, i]
        for f in (self.lib.orc_fold_probed, self.lib.orc_enumerate_probed):
            f.restype = i
            f.argtypes = [vp, C.c_char_p, i, i, vp, vp, vp, vp, vp, i, vp]
        self.lib.orc_fold_soft.restype = i
        self.lib.orc_fold_soft.argtypes = [vp, C.c_char_p, i, i, vp, vp, vp, vp, i, vp]
        self._model = model
        self.P = self.lib.orc_params_new(C.addressof(model))

    def maxloop(self, m):
        self.lib.orc_set_maxloop(self.P, m)

    def _call(self, f, seq, cp, allow, E, U, max_w, soft=False):
        n = len(seq)
        pr, up, lz = np.zeros((n + 1, n + 1)), np.zeros((n, max(max_w, 1))), C.c_double()
        a, ap = _ptr(allow, np.uint8)
        e, ep = _ptr(E, np.int32)
        u, upp = _ptr(U, np.int32)
        args = [self.P, seq.encode(), n, cp, ap, ep] + ([] if soft else [upp])
        assert f(*args, pr.ctypes.data, up.ctypes.data, max_w, C.byref(lz)) == 0
        return pr, (up if max_w > 0 else None), lz.value

    def fold(self, seq, cp=0, allow=None, E=None, U=None, max_w=0):
        return self._call(self.lib.orc_fold_probed, seq, cp, allow, E, U, max_w)

    def enumerate(self, seq, cp=0, allow=None, E=None, U=None, max_w=0):
        return self._call(self.lib.orc_enumerate_probed, seq, cp, allow, E, U, max_w)

    def fold_soft(self, seq, cp=0, allow=None, E=None, max_w=0):
        return self._call(self.lib.orc_fold_soft, seq, cp, allow, E, None, max_w, soft=True)


def _oracle_so(tmp_path_factory):
    so = tmp_path_factory.mktemp("porc") / "liboracle_probed.so"
    _cc(["gcc", "-O3", "-fPIC", "-shared", "-I", str(ROOT / "include"), str(ROOT / "tests" / "cpp" / "oracle_probed.c"),
         "-o", str(so), "-lm"])
    return so


@pytest.fixture(scope="module")
def orc_so(tmp_path_factory):
    return _oracle_so(tmp_path_factory)


@pytest.fixture(scope="module")
def porc(orc_so, model):
    o = ProbedOracle(orc_so, model)
    yield o
    o.maxloop(30)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = tmp_path_factory.mktemp("ushim") / "libunpaired_shim.so"
    csrc = ROOT / "ractip_b200" / "csrc"
    _cc(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", str(ROOT / "include"), "-I", str(csrc),
         str(csrc / "plan.cpp"), str(ROOT / "tests" / "cpp" / "unpaired_shim.cpp"), "-o", str(so)])
    lib = C.CDLL(str(so))
    vp = C.c_void_p
    lib.unpaired_shim.argtypes = [vp, vp, vp, vp, C.c_int, vp, C.c_char_p, C.c_int, vp, vp, vp, C.c_int, vp, vp]
    lib.unpaired_shim.restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def kemul(tmp_path_factory):
    so = tmp_path_factory.mktemp("uemul") / "libemul_probed.so"
    d = ROOT / "tests" / "emul"
    _cc(["g++", "-O2", "-U_FORTIFY_SOURCE", "-std=c++17", "-fPIC", "-shared", "-I", str(ROOT / "ractip_b200" / "csrc"),
         "-I", str(ROOT / "include"), "-o", str(so), str(d / "emul_probed.cpp"),
         str(ROOT / "ractip_b200" / "csrc" / "dev_model.cpp")])
    lib = C.CDLL(str(so))
    vp, i = C.c_void_p, C.c_int
    lib.emul_probed_problem.argtypes = [i, i, i, vp, C.c_double, vp, vp, vp, C.c_char_p, i, i, i, i, i, i, C.c_float, i,
                                        vp, vp, vp, vp, C.c_uint64, i, vp]
    lib.emul_probed_problem.restype = i
    return lib


def opts(**kw):
    o = dict(max_w=15, min_w=5, th_ss=0.5, th_hy=0.1, th_ac=0.003, use_pf_duplex=0)
    o.update(kw)
    return RpOpts(**o)


# ---------------------------------------------------------------------- probed oracle vs enumeration (CPU)
def _check_enum(porc, seq, cp, allow, E, U, max_w):
    pr, up, lz = porc.fold(seq, cp, allow, E, U, max_w)
    epr, eup, elz = porc.enumerate(seq, cp, allow, E, U, max_w)
    assert abs(lz - elz) < 1e-12 * max(1.0, abs(elz))
    np.testing.assert_allclose(pr, epr, rtol=0, atol=1e-12)
    if max_w:
        np.testing.assert_allclose(up, eup, rtol=0, atol=1e-12)
    return lz


@pytest.mark.parametrize("maxloop", [30, 3])
def test_probed_oracle_single_strand(porc, maxloop):
    porc.maxloop(maxloop)
    try:
        rng = np.random.default_rng(151)
        moved = 0
        for k in range(8):
            n = int(rng.integers(11, 15))
            s = rand_seq(rng, n) if k else "GGGGAAACCCCAGG"[:n]
            U = random_unpaired(rng, n)
            E = random_unpaired(rng, n) if k % 4 >= 2 else None   # with stacking pseudo-energies too
            allow = None
            if k % 2:
                m, bp, unp = problem_view(random_constraint(rng, n, 0)[0], None, n, 0, 0)
                allow = allowed_matrix(m, bp, unp)
            _check_enum(porc, s, 0, allow, E, U, 6)
            pr0 = porc.fold(s, 0, allow, E, None, 0)[0]
            moved += np.abs(porc.fold(s, 0, allow, E, U, 0)[0] - pr0).max() > 1e-6
        assert moved >= 4   # the energies do change the ensembles
    finally:
        porc.maxloop(30)


@pytest.mark.parametrize("maxloop", [30, 3])
def test_probed_oracle_two_strands(porc, maxloop):
    porc.maxloop(maxloop)
    try:
        rng = np.random.default_rng(152)
        cases = [("GGGAAUCC", "GGAUUCC"), ("GCGCAAAG", "CUUUGC")]
        for _ in range(5):
            n1, n2 = int(rng.integers(5, 8)), int(rng.integers(5, 8))
            cases.append((rand_seq(rng, n1), rand_seq(rng, n2)))
        for k, (s1, s2) in enumerate(cases):
            n1, n2 = len(s1), len(s2)
            U = random_unpaired(rng, n1 + n2)
            E = random_unpaired(rng, n1 + n2) if k % 4 >= 2 else None
            allow = None
            if k % 2:
                m, bp, unp = problem_view(*random_constraint(rng, n1, n2), n1, n2, 2)
                allow = allowed_matrix(m, bp, unp)
            _check_enum(porc, s1 + s2, n1 + 1, allow, E, U, 0)
    finally:
        porc.maxloop(30)


def test_probed_oracle_zero_data_is_bitwise_the_soft_oracle(porc):
    rng = np.random.default_rng(153)
    for n, cp in ((40, 0), (30, 17)):
        s = rand_seq(rng, n)
        w = 8 if cp == 0 else 0
        E = random_unpaired(rng, n)
        for U in (None, np.zeros(n, dtype=np.int32)):
            for e in (None, E):
                a = porc.fold(s, cp, None, e, U, w)
                b = porc.fold_soft(s, cp, None, e, w)
                assert a[2] == b[2] and np.array_equal(a[0], b[0]) and (w == 0 or np.array_equal(a[1], b[1]))


# --------------------------------------------------------------------------------------- planning (CPU)
def plan(shim, pairs, unpaired, cons=None, stack=None, o=None):
    """(rc, message, pair factors, log-Z terms, per-problem (seq_off, n, constrained, general), same plan as without)"""
    keep = []
    arr = (RpPair * len(pairs))()
    uarr = (RpUnpairedEnergy * len(pairs))()
    sarr = (RpStackEnergy * len(pairs))() if stack else None
    carr = (RpConstraint * len(pairs))() if cons else None
    for k, (s1, s2) in enumerate(pairs):
        b = [s1.encode(), s2.encode()]
        keep.append(b)
        arr[k].s1, arr[k].n1, arr[k].s2, arr[k].n2 = b[0], len(s1), b[1] or None, len(s2)
        for vec, struct, name in ((unpaired, uarr, "u"), (stack, sarr, "e")):
            if vec is None or vec[k] is None:
                continue
            for s, e in enumerate(vec[k]):
                if e is not None:
                    a = np.ascontiguousarray(e, dtype=np.float64)
                    keep.append(a)
                    setattr(struct[k], f"{name}{s + 1}", a.ctypes.data)
        if cons:
            c = [x.encode() if x is not None else None for x in cons[k]]
            keep.append(c)
            carr[k].c1, carr[k].c2 = c
    cap = sum(2 * (len(a) + len(b)) + 4 for a, b in pairs) + 16
    unp = np.zeros(cap)
    lz = np.zeros(cap)
    ulen = C.c_longlong()
    probs = np.zeros((3 * len(pairs), 4), dtype=np.int64)
    msg = C.create_string_buffer(400)
    same = C.c_int()
    rc = shim.unpaired_shim(arr, carr, sarr, uarr, len(pairs), C.byref(o or opts()), msg, 400, unp.ctypes.data,
                            C.byref(ulen), lz.ctypes.data, cap, probs.ctypes.data, C.byref(same))
    return rc, msg.value.decode(), unp[:ulen.value], lz[:3 * len(pairs)], probs, bool(same.value)


def test_plan_flags_routes_and_factors(shim):
    rng = np.random.default_rng(161)
    pairs = [("ACGU" * 18, "ACGU" * 34)] * 4
    u1 = rng.normal(0, 0.5, 72)
    u2 = rng.normal(0, 0.5, 136)
    rc, msg, unp, lz, probs, _ = plan(shim, pairs, [None, (u1, None), (None, u2), (np.zeros(72), np.zeros(136))])
    assert rc == 0, msg
    U = CON_UNPAIRED
    assert probs[:, 2].tolist() == [0, 0, 0, U, 0, U, 0, U, U, 0, 0, 0]
    assert probs[:, 3].tolist() == [0, 0, 0, 1, 0, 1, 0, 1, 1, 0, 0, 0]   # band kernel without data
    g1, g2 = np.exp(dcal(u1) * 10.0 / KT), np.exp(dcal(u2) * 10.0 / KT)
    off = {k: int(probs[k, 0]) for k in range(12)}
    close = lambda a, b: np.testing.assert_allclose(a, b, rtol=1e-15, atol=0)
    close(unp[off[3]:off[3] + 72], g1)
    close(unp[off[5]:off[5] + 208], np.concatenate([g1, np.ones(136)]))
    close(unp[off[7]:off[7] + 136], g2)
    close(unp[off[8]:off[8] + 208], np.concatenate([np.ones(72), g2]))
    others = np.ones(len(unp), dtype=bool)
    for k, m in ((3, 72), (5, 208), (7, 136), (8, 208)):
        others[off[k]:off[k] + m] = False
    assert np.all(unp[others] == 1.0)
    l1, l2 = -dcal(u1).sum() * 10.0 / KT, -dcal(u2).sum() * 10.0 / KT
    np.testing.assert_allclose(lz[3:9], [l1, 0, l1, 0, l2, l2], rtol=1e-13, atol=1e-13)
    # with -c keys and stacking energies on the same pair: all bits, one route
    cons = [(None, None), ("(" + "." * 70 + ")", None), (None, None), (None, None)]
    e1 = rng.normal(0, 1, 72)
    rc, msg, _, _, probs, _ = plan(shim, pairs, [None, (u1, None), None, None], cons, [None, (e1, None), None, None])
    assert rc == 0, msg
    assert probs[3:6, 2].tolist() == [CON_KEYS | CON_STACK | U, 0, CON_KEYS | CON_STACK | U]
    assert probs[3:6, 3].tolist() == [1, 0, 1]


def test_plan_duplex_ignores_the_data(shim):
    pairs = [("ACGU" * 18, "ACGU" * 34)]
    u = (np.full(72, 0.3), np.full(136, -0.3))
    rc, msg, _, _, probs, _ = plan(shim, pairs, [u], o=opts(use_pf_duplex=1))
    assert rc == 0, msg
    assert probs[:, 2].tolist() == [CON_UNPAIRED, CON_UNPAIRED, 0] and probs[2, 3] == 1   # duplex_kernel's queue
    # the range check does not count a co-fold that --duplex does not run
    big = (np.full(72, 2.0), np.full(136, 0.3))   # B(s1) = 72 * 200 * 10 / kT = 233, B(s1) + B(s2) = 299 + ... < 345
    big2 = (np.full(72, 2.0), np.full(136, 0.9))  # B(s1) + B(s2) = 233 + 199 > 345; each alone < 345
    assert plan(shim, pairs, [big2], o=opts(use_pf_duplex=1))[0] == 0
    rc, msg, *_ = plan(shim, pairs, [big2])
    assert rc == RP_ERR_UNSUPPORTED and msg.startswith("pair 0, problem s1&s2:"), msg
    assert plan(shim, pairs, [big])[0] == 0


def test_plan_without_data_is_the_plain_plan(shim):
    pairs = [("ACGU" * 18, "ACGU" * 34), ("GGGAAACCC" * 3, "")]
    cons = [("(" + "." * 70 + ")", None), (None, None)]
    stack = [(np.linspace(-1, 1, 72), None), None]
    for unpaired in ([None, None], [(None, None), (None, None)],
                     [(np.zeros(72), np.zeros(136)), (np.full(27, 0.0049), None)],
                     [(np.full(72, -0.00499), None), (np.zeros(27), None)]):
        for c, st in ((None, None), (cons, None), (None, stack), (cons, stack)):
            rc, msg, unp, lz, probs, same = plan(shim, pairs, unpaired, c, st)
            assert rc == 0, msg
            assert len(unp) == 0 and same and not (probs[:, 2] & CON_UNPAIRED).any()


def test_plan_rounding_boundary(shim):
    pairs = [("GGGAAACCC", "")]
    u = np.array([0.005, -0.005, 0.0049999, -0.0049999, 0.015, -0.025, 1.234, 0.0, 0.0])
    rc, msg, unp, lz, probs, same = plan(shim, pairs, [(u, None)])
    assert rc == 0 and probs[0, 2] == CON_UNPAIRED and not same
    want = np.array([1, -1, 0, 0, 2, -3, 123, 0, 0])
    off = int(probs[0, 0])
    np.testing.assert_allclose(unp[off:off + 9], np.exp(want * 10.0 / KT), rtol=1e-15, atol=0)
    assert np.count_nonzero(unp[off:off + 9] == 1.0) == 4
    np.testing.assert_array_equal(dcal(u), want)
    assert abs(lz[0] - (-want.sum() * 10.0 / KT)) < 1e-14


@pytest.mark.parametrize("bad,where", [
    (float("nan"), "pair 1, u2, position 3: nan kcal/mol is not finite"),
    (float("inf"), "pair 1, u2, position 3: inf kcal/mol is not finite"),
    (float("-inf"), "pair 1, u2, position 3: -inf kcal/mol is not finite")])
def test_non_finite_energies(shim, bad, where):
    u2 = np.zeros(4)
    u2[2] = bad
    rc, msg, *_ = plan(shim, [("ACGU" * 5, "ACGU"), ("GGGAAACCC", "GGGU")], [(np.ones(20), None), (None, u2)])
    assert rc == RP_ERR_ARG and msg == where


def test_range_check_at_the_limit(shim):
    """B = sum |E| 10 / kT after rounding: just below ln 10^150 is planned, just above is RP_ERR_UNSUPPORTED"""
    per = 10.0 / KT   # B of one base at 0.01 kcal/mol
    units = int(MAX_B / per)   # the largest total of |E| (0.01 kcal/mol) inside the range
    assert units * per <= MAX_B < (units + 1) * per
    n = 400
    base, extra = divmod(units, n)
    E = np.full(n, base, dtype=np.int64)
    E[:extra] += 1
    E[1::2] *= -1   # the sign does not matter
    s = rand_seq(np.random.default_rng(171), n)
    u = E / 100.0
    rc, msg, _, _, probs, _ = plan(shim, [("GGGAAACCC", ""), (s, "")], [None, (u, None)])
    assert rc == 0 and probs[3, 2] == CON_UNPAIRED, msg
    u2 = u.copy()
    u2[-1] += 0.01 * np.sign(u2[-1])   # one more 0.01 kcal/mol
    rc, msg, *_ = plan(shim, [("GGGAAACCC", ""), (s, "")], [None, (u2, None)])
    assert rc == RP_ERR_UNSUPPORTED, msg
    m = re.match(r"pair 1, problem s1: the unpaired pseudo-energies give B = sum \|E\| / kT = ([0-9.]+), beyond ln "
                 r"10\^150 = 345\.39", msg)
    assert m and abs(float(m.group(1)) - (units + 1) * per) < 0.006, msg
    # rounding first: values that round to 0 add nothing
    rc, *_ = plan(shim, [(s, "")], [(np.where(u == 0, 0.0049, u), None)])
    assert rc == 0


# ------------------------------------------------------------------------------------------ emulator (CPU)
def _emul(kemul, model, U, seq, cp, kind, max_w, n1, n2, route, G, lockstep, E=None, keys=None, num=0, seed=5, T=64):
    n = len(seq)
    bp = np.zeros((n + 1) * (n + 2) // 2, dtype=np.float32)
    up = np.zeros((n, max(max_w, 1)), dtype=np.float32)
    hp = np.zeros((n1 + 1, n2 + 1), dtype=np.float32)
    smp = np.zeros((max(num, 1), n), dtype=np.int16)
    lz = C.c_double()
    upf = None if U is None else np.ascontiguousarray(np.concatenate([[1.0], np.exp(np.asarray(U) * 10.0 / KT)]))
    ulz = 0.0 if U is None else float(-np.sum(U) * 10.0 / KT)
    stk = None if E is None else np.ascontiguousarray(np.concatenate([[1.0], np.exp(-np.asarray(E) * 10.0 / KT)]))
    key = None if keys is None else np.ascontiguousarray(keys, dtype=np.uint16)
    rc = kemul.emul_probed_problem(route, G, int(lockstep), None if upf is None else upf.ctypes.data, ulz,
                                   None if stk is None else stk.ctypes.data, None if key is None else key.ctypes.data,
                                   C.addressof(model), seq.encode(), n, cp, kind, max_w, n1, n2, 0.1, T,
                                   bp.ctypes.data, up.ctypes.data, hp.ctypes.data, C.byref(lz), seed, num,
                                   smp.ctypes.data)
    assert rc == 0, rc
    return bp, up, hp, lz.value, smp[:num]


@pytest.mark.parametrize("lockstep", [False, True])
def test_emulator_routes(kemul, porc, model, lockstep):
    """bp, up and hp of every general route against the literal oracle (the fp32 outputs round the same doubles, so
    they agree to fp32 rounding), log Z within 1e-9"""
    rng = np.random.default_rng(171)
    s1, s2 = rand_seq(rng, 47), rand_seq(rng, 38)
    U1, U2 = random_unpaired(rng, 47), random_unpaired(rng, 38)
    E1 = random_unpaired(rng, 47)
    pr1, up1, lz1 = porc.fold(s1, 0, None, E1, U1, 8)
    pr12, _, lz12 = porc.fold(s1 + s2, 48, None, None, np.concatenate([U1, U2]), 0)
    assert abs(lz1 - porc.fold(s1, 0, None, E1, None, 0)[2]) > 1.0   # the data move log Z
    want = np.zeros((48, 39))
    want[1:, 1:] = pr12[1:48, 48:]
    want = np.where((want >= 0.1) & (want.astype(np.float32) > np.float32(0.1)), want, 0)
    for route, G in ROUTES:
        b, u, _, lz, _ = _emul(kemul, model, U1, s1, 0, 0, 8, 47, 0, route, G, lockstep, E=E1)
        B = _bp_matrix(b, 47)
        np.testing.assert_allclose(B, pr1.astype(np.float32), rtol=1e-6, atol=1e-30)
        np.testing.assert_allclose(u, up1.astype(np.float32), rtol=1e-6, atol=1e-30)
        assert abs(lz - lz1) < 1e-9, (route, G)
        _, _, h, lz, _ = _emul(kemul, model, np.concatenate([U1, U2]), s1 + s2, 48, 1, 0, 47, 38, route, G, lockstep)
        np.testing.assert_allclose(h, want.astype(np.float32), rtol=1e-6, atol=1e-30)
        assert abs(lz - lz12) < 1e-9, (route, G)


def test_emulator_log_z_in_double(kemul, porc, model):
    """log Z, the one output kept in fp64, within 1e-12 relative of the literal oracle on every route"""
    rng = np.random.default_rng(172)
    s = rand_seq(rng, 60)
    U = random_unpaired(rng, 60)
    _, _, lz_o = porc.fold(s, 0, None, None, U, 0)
    for route, G in ROUTES:
        _, _, _, lz, _ = _emul(kemul, model, U, s, 0, 0, 8, 60, 0, route, G, True)
        assert abs(lz - lz_o) <= 1e-12 * abs(lz_o) + 1e-12


# ------------------------------------------------------------------------------------------ sampling (CPU)
@pytest.fixture(scope="module")
def model0(lib):
    """the default model with the clipped tables (pf_smooth = 0) that the integer energy evaluation uses"""
    from ractip_b200 import default_model
    m = default_model()
    m.pf_smooth = 0
    return m


def exact_distribution(model0, porc0, seq, cp, U):
    """{pair table bytes: probability} from the integer energy evaluation plus the unpaired pseudo-energies of each
    structure's unpaired bases (and intermolecular pairs' bases), over the probed oracle's Z"""
    from ractip_b200 import energy_of_structure
    n = len(seq)
    _, _, logz = porc0.fold(seq, cp, None, None, U, 0)
    kT = KT / 1000.0
    out = {}
    for pairs in all_structures(n):
        if not all(can_pair(seq[i - 1], seq[j - 1]) for i, j in pairs):
            continue
        e = energy_of_structure(model0, seq, to_string(n, pairs), cp if cp else -1)
        if cp and any(i < cp <= j for i, j in pairs):
            e -= model0.DuplexInit37 / 100.0
        paired = {x for i, j in pairs if not (cp and i < cp <= j) for x in (i, j)}
        e += sum(int(U[x - 1]) for x in range(1, n + 1) if x not in paired) / 100.0
        t = np.zeros(n, dtype=np.int16)
        for i, j in pairs:
            t[i - 1], t[j - 1] = j, i
        out[t.tobytes()] = math.exp(-e / kT - logz)
    assert abs(sum(out.values()) - 1.0) < 1e-3
    return out


def check_distribution(tables, exact):
    """the statistical test of tests/test_sampling.py"""
    N = len(tables)
    counts = {}
    for t in tables:
        counts[t.tobytes()] = counts.get(t.tobytes(), 0) + 1
    assert set(counts) <= set(exact), "a sample outside the ensemble"
    for k, p in exact.items():
        if N * p >= 20:
            c = counts.get(k, 0)
            assert abs(c - N * p) <= 6 * math.sqrt(N * p * (1 - p)), (c, N * p)
    tvd = 0.5 * sum(abs(counts.get(k, 0) / N - p) for k, p in exact.items())
    bound = 3 * 0.5 * sum(math.sqrt(p / N) for p in exact.values())
    assert tvd < bound, (tvd, bound)


SAMPLE_CASES = [("GGGAAACCCAGC", 0), ("GGCAUCCG", 0), ("GGGAAC", 7)]


@pytest.mark.parametrize("seq,cp", SAMPLE_CASES)
def test_emulator_samples_match_exact_distribution(kemul, orc_so, model0, seq, cp):
    porc0 = ProbedOracle(orc_so, model0)
    rng = np.random.default_rng(181 + len(seq))
    if cp:
        seq = seq + "GUUCCC"
    n = len(seq)
    U = random_unpaired(rng, n, scale=120)
    exact = exact_distribution(model0, porc0, seq, cp, U)
    kind = 1 if cp else 0
    n1, n2 = (cp - 1, n - cp + 1) if cp else (n, 0)
    _, _, _, _, smp = _emul(kemul, model0, U, seq, cp, kind, 0, n1, n2, 10, 1, True, num=20000, seed=7)
    check_distribution(smp, exact)


# ------------------------------------------------------------------------------------------ front end (CPU)
def test_read_shape_under_w(tmp_path, lib):
    from ractip_b200.frontend import read_shape
    p = tmp_path / "u.dat"
    p.write_text("1 G 0.5\n3 -1.25\n6 U 0.0\n")
    r = read_shape(str(p), "GGGAAU")
    assert r[0] == 0.5 and r[2] == -1.25 and r[5] == 0.0 and np.isnan(r[1]) and np.isnan(r[4])


def test_predict_passes_unpaired_energies_and_leaves_shuffles_bare(monkeypatch):
    from ractip_b200 import frontend
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
    r = np.array([0.1, -0.2, np.nan, 0.4, 1.5, 0, 0, -2, 3])
    with pytest.raises(Stop):
        frontend.predict(FakeStage(), [(a, b)], zscore=12, num_shuffling=3, shape={"b": r}, shape_slope=2.0,
                         shape_method="W")
    (u1, u2), = calls[0][2]["unpaired_energies"]
    assert u1 is None and np.array_equal(u2, np.nan_to_num(r, nan=0.0))
    assert "stack_energies" not in calls[0][2]
    assert len(calls[1][0]) == 3 and calls[1][2] == {}
    with pytest.raises(ValueError, match="shape method 'X': expected D or W"):
        frontend.predict(FakeStage(), [(a, b)], shape={"b": r}, shape_method="X")


def _cli(args, cwd=ROOT):
    return subprocess.run([sys.executable, "-m", "ractip_b200"] + args, cwd=cwd, stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True, timeout=600)


def test_command_line_input_errors(tmp_path, lib, bundled):
    seqs = bundled["sequences"]
    (tmp_path / "a.fa").write_text(f">MicA\n{seqs['MicA']}\n")
    (tmp_path / "b.fa").write_text(f">ompA\n{seqs['ompA']}\n")
    (tmp_path / "ok.dat").write_text("1 0.5\n")
    (tmp_path / "bad.dat").write_text(f"{len(seqs['MicA']) + 1} -0.5\n")
    fa = [str(tmp_path / "a.fa"), str(tmp_path / "b.fa")]
    for extra, msg in ((["--shape-method", "Z"], "--shape-method Z: expected D or W"),
                       (["--shape", f"MicA={tmp_path / 'ok.dat'}", "--shape-method", "w"], "expected D or W"),
                       (["--shape", f"MicA={tmp_path / 'bad.dat'}", "--shape-method", "W"], "is outside 1..72"),
                       (["--shape", f"SodB={tmp_path / 'ok.dat'}", "--shape-method", "W"], "no record named 'SodB'")):
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


def _oracle_pair(porc, s1, s2, u1, u2, o, c1=None, c2=None, e1=None, e2=None):
    """the probed oracle's (pr, up, logZ) of the three problems, from kcal/mol energies as the library takes them"""
    n1, n2 = len(s1), len(s2)
    z = lambda v, m: dcal(v) if v is not None else np.zeros(m, dtype=np.int64)
    U1, U2, E1, E2 = z(u1, n1), z(u2, n2), z(e1, n1), z(e2, n2)
    out = {}
    for which, seq, U, E in ((0, s1, U1, E1), (1, s2, U2, E2), (2, s1 + s2, np.concatenate([U1, U2]),
                                                              np.concatenate([E1, E2]))):
        A = None
        if c1 is not None or c2 is not None:
            m, bp, unp = problem_view(c1, c2, n1, n2, which)
            A = allowed_matrix(m, bp, unp)
        out[which] = porc.fold(seq, n1 + 1 if which == 2 else 0, A, E, U, 0 if which == 2 else o.max_w)
    return out


def _hp_want(pr, n1, n2, th):
    want = np.zeros((n1 + 1, n2 + 1))
    want[1:, 1:] = pr[1:n1 + 1, n1 + 1:]
    return np.where((want >= th) & (want.astype(np.float32) > np.float32(th)), want, 0)


def _sets(M, th):
    return set(zip(*np.nonzero(M > th)))


def _compare(r, lz, orc, n1, n2, o):
    for which, (bp, nn, up) in ((0, (r.bp1, n1, r.up1)), (1, (r.bp2, n2, r.up2))):
        pr, oup, olz = orc[which]
        B = _bp_matrix(bp, nn)
        np.testing.assert_allclose(B, pr, rtol=0, atol=TOL)
        np.testing.assert_allclose(up, oup, rtol=0, atol=TOL)
        assert _sets(B, o.th_ss) == _sets(pr.astype(np.float32), o.th_ss)   # the IP's x / y variables
        assert _sets(up, o.th_ac) == _sets(oup.astype(np.float32), o.th_ac)   # its v / w
        assert abs(lz[which] - olz) < 1e-9
    pr, _, olz = orc[2]
    want = _hp_want(pr, n1, n2, o.th_hy)
    np.testing.assert_allclose(r.hp, want, rtol=0, atol=TOL)
    assert _sets(r.hp, o.th_hy) == _sets(want.astype(np.float32), o.th_hy)   # its z
    assert abs(lz[2] - olz) < 1e-9


def _run(stage, pairs, o, cons=None, stack=None, unpaired=None, samples=0, seed=1):
    b = stage.batch(pairs, o, cons, stack, samples=samples, sample_seed=seed, unpaired_energies=unpaired)
    try:
        b.run()
        flat = b.fetch_dense()
        smp = b.fetch_samples() if samples else None
        return b.split_dense(flat), b.fetch_logz(), flat.copy(), smp
    finally:
        b.close()


def _bundled_unpaired(bundled):
    seqs = bundled["sequences"]
    rng = np.random.default_rng(191)
    pairs = [(seqs[a], seqs[b]) for a, b in bundled["pairs"]]
    return pairs, [(random_kcal(rng, len(s1), 0.3), random_kcal(rng, len(s2), 0.3)) for s1, s2 in pairs]


@gpu
@pytest.mark.parametrize("env", [{}, {"RP_BAND": "0"}], ids=["default", "no_band"])
def test_gpu_bundled_pairs(porc, bundled, monkeypatch, env):
    pairs, unpaired = _bundled_unpaired(bundled)
    o = opts()
    stage = _stage_env(monkeypatch, env)
    try:
        res, lz, _, _ = _run(stage, pairs, o, unpaired=unpaired)
        for (s1, s2), (u1, u2), r, z in zip(pairs, unpaired, res, lz):
            _compare(r, z, _oracle_pair(porc, s1, s2, u1, u2, o), len(s1), len(s2), o)
        # sparse lists and tensors of the probed batch agree with its dense fetch
        recs = stage.run_sparse(pairs, o, unpaired_energies=unpaired)
        for (s1, s2), r, sp in zip(pairs, res, recs):
            n1, n2 = len(s1), len(s2)
            P1 = _bp_matrix(r.bp1, n1)
            want_x = sorted((i - 1, j - 1) for i in range(1, n1 + 1) for j in range(i + 1, n1 + 1) if P1[i, j] > o.th_ss)
            assert sorted((int(x["i"]), int(x["j"])) for x in sp.x) == want_x
            want_z = sorted((i - 1, j - 1) for i in range(1, n1 + 1) for j in range(1, n2 + 1) if r.hp[i, j] > o.th_hy)
            assert sorted((int(x["i"]), int(x["j"])) for x in sp.z) == want_z
        dense = stage.run_dense(pairs, o, unpaired_energies=unpaired)
        for r, d in zip(res, dense):
            assert r.bp1.tobytes() == d.bp1.tobytes() and r.hp.tobytes() == d.hp.tobytes()
        import torch
        b = stage.batch(pairs, o, unpaired_energies=unpaired)
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


def _long_case(porc, dis):
    """620x300 and 720x90 pairs with unpaired and stacking pseudo-energies and -c lines (B inside the range)"""
    if not _LONG:
        rng = np.random.default_rng(192)
        o = opts()
        pairs = [(rand_seq(rng, 620), rand_seq(rng, 300)), (rand_seq(rng, 720), rand_seq(rng, 90))]
        unpaired = [(random_kcal(rng, len(a), 0.12), random_kcal(rng, len(b), 0.12)) for a, b in pairs]
        stack = [(random_kcal(rng, 620, 0.8), None), (None, random_kcal(rng, 90, 0.8))]
        cons = [random_constraint(rng, 620, 300, dens=0.05), random_constraint(rng, 720, 90, dens=0.05)]
        orc = [_oracle_pair(porc, a, b, u1, u2, o, c1, c2, e1, e2)
               for (a, b), (u1, u2), (c1, c2), (e1, e2) in zip(pairs, unpaired, cons, stack)]
        _LONG["case"] = (pairs, unpaired, stack, cons, orc)
    return _LONG["case"]


@gpu
@pytest.mark.parametrize("env", ROUTE_ENVS, ids=["default", "wide", "cluster8", "cluster16"])
def test_gpu_long_pair_routes(porc, bundled, kemul, model, monkeypatch, env):
    pairs, unpaired, stack, cons, orc = _long_case(porc, bundled["readme_dis"])
    o = opts()
    stage = _stage_env(monkeypatch, env)
    try:
        res, lz, _, smp = _run(stage, pairs, o, cons, stack, unpaired, samples=4, seed=11)
    finally:
        stage.close()
    for (s1, s2), r, z, oc in zip(pairs, res, lz, orc):
        _compare(r, z, oc, len(s1), len(s2), o)
    for d, (s1, s2) in zip(smp, pairs):
        for key, n in (("s1", len(s1)), ("s2", len(s2)), ("co", len(s1) + len(s2))):
            t = d[key]
            assert t.shape == (4, n)
            for row in t:   # valid pair tables
                nz = np.nonzero(row)[0]
                assert np.all(row[row[nz] - 1] == nz + 1)


@gpu
def test_gpu_samples_equal_the_emulator(kemul, model, bundled, monkeypatch):
    seqs = bundled["sequences"]
    s1, s2 = seqs["MicA"], seqs["ompA"]
    rng = np.random.default_rng(193)
    u1, u2 = random_kcal(rng, len(s1), 0.4), random_kcal(rng, len(s2), 0.4)
    o = opts()
    stage = _stage_env(monkeypatch, {})
    try:
        _, _, _, smp = _run(stage, [(s1, s2)], o, unpaired=[(u1, u2)], samples=16, seed=3)
    finally:
        stage.close()
    U1, U2 = dcal(u1), dcal(u2)
    for which, seq, cp, U, kind, n1, n2 in (("s1", s1, 0, U1, 0, len(s1), 0),
                                            ("co", s1 + s2, len(s1) + 1, np.concatenate([U1, U2]), 1, len(s1), len(s2))):
        # pair 0 of the batch: the emulator binds pair 0 and problem kind == 1 ? 2 : 0
        _, _, _, _, e = _emul(kemul, model, U, seq, cp, kind, 0, n1, n2, 0, 1, True, num=16, seed=3)
        assert np.array_equal(smp[0][which], e), which


@gpu
def test_gpu_byte_identity(bundled, monkeypatch):
    seqs, dis = bundled["sequences"], bundled["readme_dis"]
    pairs = [(seqs[a], seqs[b]) for a, b in (("MicA", "ompA"), ("DIS", "DIS"), ("OxyS", "fhlA"))]
    o = opts()
    rng = np.random.default_rng(194)
    stage = _stage_env(monkeypatch, {})
    try:
        # all-zero data: none
        _, lz0, plain, _ = _run(stage, pairs, o)
        zero = [(np.zeros(len(a)), np.full(len(b), 0.004)) for a, b in pairs]
        _, lz1, flat, _ = _run(stage, pairs, o, unpaired=zero)
        assert plain.tobytes() == flat.tobytes() and lz0.tobytes() == lz1.tobytes()
        # the unprobed pairs of a mixed batch against the same pairs alone
        probed = (random_kcal(rng, len(pairs[0][0])), None)
        r1, lz1, _, _ = _run(stage, pairs, o, unpaired=[probed, None, (None, None)])
        r0, lz0, _, _ = _run(stage, pairs[1:], o)
        for k in (1, 2):
            for f in ("bp1", "bp2", "up1", "up2", "hp"):
                assert getattr(r1[k], f).tobytes() == getattr(r0[k - 1], f).tobytes()
            assert lz1[k].tobytes() == lz0[k - 1].tobytes()
        assert r1[0].bp1.tobytes() != _run(stage, pairs[:1], o)[0][0].bp1.tobytes()   # the data did reach pair 0
        # --duplex: the hybridization ignores the data
        od = opts(use_pf_duplex=1)
        d0, _, _, _ = _run(stage, pairs, od)
        both = [(random_kcal(rng, len(a)), random_kcal(rng, len(b))) for a, b in pairs]
        d1, _, _, _ = _run(stage, pairs, od, unpaired=both)
        for k in range(3):
            assert d0[k].hp.tobytes() == d1[k].hp.tobytes()
        # batches with only constraints or only stacking energies: the same bytes with ue == NULL as before
        cons = [None, (dis["s1"], dis["s2"]), None]
        stack = [(random_kcal(rng, len(a), 1.0), None) for a, b in pairs]
        for c, st in ((cons, None), (None, stack), (cons, stack)):
            _, lza, fa, _ = _run(stage, pairs, o, c, st)
            _, lzb, fb, _ = _run(stage, pairs, o, c, st, unpaired=[None] * 3)
            _, lzc, fc, _ = _run(stage, pairs, o, c, st, unpaired=zero)
            assert fa.tobytes() == fb.tobytes() == fc.tobytes() and lza.tobytes() == lzb.tobytes() == lzc.tobytes()
    finally:
        stage.close()


def _pack_bp(pr, n):
    bp = np.zeros((n + 1) * (n + 2) // 2, dtype=np.float32)
    for i in range(1, n + 1):
        off = i * (2 * n + 1 - i) // 2
        bp[off + i + 1:off + n + 1] = pr[i, i + 1:]
    return bp


@gpu
def test_gpu_command_line(porc, model, bundled, tmp_path):
    from ractip_b200 import bp_offsets, default_ip_opts, solve_joint
    from ractip_b200.frontend import read_shape
    from ractip_b200.stage import PairProbabilities
    seqs = bundled["sequences"]
    s1, s2 = seqs["MicA"], seqs["ompA"]
    rng = np.random.default_rng(195)
    (tmp_path / "a.fa").write_text(f">MicA\n{s1}\n")
    (tmp_path / "b.fa").write_text(f">ompA\n{s2}\n")
    lines = [f"{i + 1} {s1[i]} {v:.2f}" for i, v in enumerate(random_kcal(rng, len(s1), 0.6)) if v != 0]
    (tmp_path / "MicA.dat").write_text("\n".join(lines) + "\n")
    r = _cli(["--shape", f"MicA={tmp_path / 'MicA.dat'}", "--shape-method", "W", str(tmp_path / "a.fa"),
              str(tmp_path / "b.fa")])
    assert r.returncode == 0, r.stdout
    out = r.stdout.splitlines()
    u1 = np.nan_to_num(read_shape(str(tmp_path / "MicA.dat"), s1), nan=0.0)
    o = opts()
    orc = _oracle_pair(porc, s1, s2, u1, None, o)
    P = PairProbabilities(_pack_bp(orc[0][0], len(s1)), bp_offsets(len(s1)), orc[0][1].astype(np.float32),
                          _pack_bp(orc[1][0], len(s2)), bp_offsets(len(s2)), orc[1][1].astype(np.float32),
                          _hp_want(orc[2][0], len(s1), len(s2), o.th_hy).astype(np.float32))
    j = solve_joint(model, s1, s2, P, default_ip_opts())
    assert out[0] == ">MicA" and out[2] == j.r1 and out[5] == j.r2, (out, j.r1, j.r2)
