"""Minimum free energy structures (rp_run_mfe): the integer Zuker kernel against a plain oracle.

The oracle (tests/cpp/oracle_mfe.c) is pinned by exhaustive enumeration of the integer energy evaluation
(rp_energy_of_structure) plus the pseudo-energy terms, computed here in Python.  CPU: the oracle, the kernel's phase
functions in the host emulator (serial and warp-lockstep, several CTA widths) against it, the host planning and its
errors, the front end's lines.  GPU: the library against the oracle and the emulator, cross-checks against the
partition function and the sampler, the command line."""
import ctypes as C
import math
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from ractip_b200._lib import RpConstraint, RpPair, RpStackEnergy, RpUnpairedEnergy

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(Path(__file__).resolve().parent))
from conftest import rand_seq  # noqa: E402
from test_constraints import allowed_matrix, problem_view, random_constraint  # noqa: E402
from test_ip import all_structures, can_pair, to_string  # noqa: E402

RP_ERR_ARG, RP_ERR_CAPACITY, RP_ERR_UNSUPPORTED, RP_INF = 1, 9, 10, 10000000
CON_KEYS, CON_STACK, CON_UNPAIRED = 1, 2, 8
KT = (37.0 + 273.15) * 1.98717
gpu = pytest.mark.gpu


def _cc(cmd):
    subprocess.run(cmd, check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)


def dcal(e):
    """kcal/mol -> integer 0.01 kcal/mol, half away from zero (the library's rounding)"""
    e = np.asarray(e, dtype=np.float64)
    return (np.sign(e) * np.floor(np.abs(e) * 100.0 + 0.5)).astype(np.int64)


def random_energies(rng, n, scale=300):
    """integer pseudo-energies (0.01 kcal/mol): many zeros, both signs, a few large ones"""
    E = rng.integers(-scale, scale, size=n)
    E[rng.random(n) < 0.3] = 0
    big = rng.random(n) < 0.08
    E[big] = rng.choice([-900, 1500, 4000], size=int(big.sum()))
    return E.astype(np.int32)


def _arr(a, dtype):
    return None if a is None else np.ascontiguousarray(a, dtype=dtype)


# ------------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope="module")
def morc(tmp_path_factory, model):
    so = tmp_path_factory.mktemp("mfeorc") / "liboracle_mfe.so"
    _cc(["gcc", "-O3", "-fPIC", "-shared", "-I", str(ROOT / "include"), str(ROOT / "tests" / "cpp" / "oracle_mfe.c"),
         "-o", str(so), "-lm"])
    lib = C.CDLL(str(so))
    vp = C.c_void_p
    lib.orc_mfe.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, vp, vp, vp, vp]
    lib.orc_mfe.restype = C.c_int

    def mfe(seq, cp=0, allow=None, E=None, U=None, m=model):
        a, e, u = _arr(allow, np.uint8), _arr(E, np.int32), _arr(U, np.int32)
        out = C.c_int()
        assert lib.orc_mfe(C.addressof(m), seq.encode(), len(seq), cp, None if a is None else a.ctypes.data,
                           None if e is None else e.ctypes.data, None if u is None else u.ctypes.data, C.byref(out)) == 0
        return out.value
    return mfe


@pytest.fixture(scope="module")
def kemul(tmp_path_factory):
    so = tmp_path_factory.mktemp("mfeemul") / "libemul_mfe.so"
    _cc(["g++", "-O2", "-U_FORTIFY_SOURCE", "-std=c++17", "-fPIC", "-shared", "-I", str(ROOT / "ractip_b200" / "csrc"),
         "-I", str(ROOT / "include"), "-o", str(so), str(ROOT / "tests" / "emul" / "emul_mfe.cpp"),
         str(ROOT / "ractip_b200" / "csrc" / "dev_model.cpp")])
    lib = C.CDLL(str(so))
    vp, i = C.c_void_p, C.c_int
    lib.emul_mfe_problem.argtypes = [i, i, vp, C.c_char_p, i, i, vp, vp, vp, vp, vp]
    lib.emul_mfe_problem.restype = i
    return lib


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = tmp_path_factory.mktemp("mfeshim") / "libmfe_shim.so"
    csrc = ROOT / "ractip_b200" / "csrc"
    _cc(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", str(ROOT / "include"), "-I", str(csrc),
         str(csrc / "plan.cpp"), str(ROOT / "tests" / "cpp" / "mfe_shim.cpp"), "-o", str(so)])
    lib = C.CDLL(str(so))
    vp = C.c_void_p
    lib.mfe_shim.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, vp, C.c_char_p, C.c_int, vp, vp, C.c_int, vp, vp, vp,
                             vp, C.c_int]
    lib.mfe_shim.restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def model0(lib):
    """the default model with the clipped tables (pf_smooth = 0) that the integer energy evaluation uses"""
    from ractip_b200 import default_model
    m = default_model()
    m.pf_smooth = 0
    return m


def emul(kemul, model, seq, cp=0, keys=None, E=None, U=None, lockstep=False, T=64):
    """(pair table, energy in 0.01 kcal/mol) of the kernel's phase functions on the host; per-base data 0-based"""
    n = len(seq)
    one = lambda a, dt: None if a is None else np.ascontiguousarray(np.concatenate([[0], np.asarray(a)]), dtype=dt)
    k, e, u = one(keys, np.uint16), one(E, np.int32), one(U, np.int32)
    pt = np.zeros(n, dtype=np.int16)
    en = C.c_int()
    rc = kemul.emul_mfe_problem(int(lockstep), T, C.addressof(model), seq.encode(), n, cp,
                                None if k is None else k.ctypes.data, None if e is None else e.ctypes.data,
                                None if u is None else u.ctypes.data, pt.ctypes.data, C.byref(en))
    assert rc == 0, rc
    return pt, en.value


# ------------------------------------------------------------------------------- energy of a structure (Python)
def pairs_of(pt):
    return [(k + 1, int(p)) for k, p in enumerate(pt) if p > k + 1]


def pseudo(pairs, n, cp, E, U):
    """stacking pseudo-energies of the stacks within one strand + unpaired pseudo-energies of the unpaired bases (a base
    paired across the nick counts as unpaired)"""
    same = lambda i, j: cp <= 0 or j < cp or i >= cp
    ps = set(pairs)
    e = 0
    if E is not None:
        for i, j in pairs:
            if (i + 1, j - 1) in ps and same(i, j):
                e += int(E[i - 1] + E[i] + E[j - 2] + E[j - 1])
    if U is not None:
        paired = {x for i, j in pairs if same(i, j) for x in (i, j)}
        e += int(sum(int(U[x - 1]) for x in range(1, n + 1) if x not in paired))
    return e


def energy(model, seq, cp, pairs, E=None, U=None):
    """E(S) of the MFE's definition in 0.01 kcal/mol: rp_energy_of_structure (DuplexInit included) plus the pseudo terms"""
    from ractip_b200 import energy_of_structure
    n = len(seq)
    e = energy_of_structure(model, seq, to_string(n, pairs), cp if cp else -1)
    return int(round(e * 100)) + pseudo(pairs, n, cp, E, U)


def check_structure(model, seq, cp, pt, e, allow=None, E=None, U=None):
    """the table is a valid structure of the ensemble, respects the constraint, and evaluates to e"""
    pairs = pairs_of(pt)
    for i, j in pairs:
        assert pt[j - 1] == i and j - i > 3 and can_pair(seq[i - 1].upper(), seq[j - 1].upper())
        if allow is not None:
            assert allow[i, j], (i, j)
    assert energy(model, seq, cp, pairs, E, U) == e


# ------------------------------------------------------------------------------ oracle vs enumeration (CPU)
def _brute(model, seq, cp, allow, E, U):
    best = None
    for pairs in all_structures(len(seq)):
        if not all(can_pair(seq[i - 1], seq[j - 1]) for i, j in pairs):
            continue
        if allow is not None and not all(allow[i, j] for i, j in pairs):
            continue
        e = energy(model, seq, cp, pairs, E, U)
        best = e if best is None else min(best, e)
    return best


def test_oracle_equals_enumeration_single_strand(morc, model):
    rng = np.random.default_rng(401)
    for k in range(14):
        n = int(rng.integers(9, 15))
        s = rand_seq(rng, n, "GCGCAU") if k else "GGGGAAACCCCAGG"[:n]
        allow = None
        if k % 3 == 1:
            m, bp, unp = problem_view(random_constraint(rng, n, 0)[0], None, n, 0, 0)
            allow = allowed_matrix(m, bp, unp)
        E = random_energies(rng, n) if k % 4 >= 2 else None
        U = random_energies(rng, n, 150) if k % 2 else None
        assert morc(s, 0, allow, E, U) == _brute(model, s, 0, allow, E, U), (s, k)


def test_oracle_equals_enumeration_two_strands(morc, model):
    rng = np.random.default_rng(402)
    cases = [("GGGAAUCC", "GGAUUCC"), ("GCGCAAAG", "CUUUGC")]
    for _ in range(10):
        cases.append((rand_seq(rng, int(rng.integers(4, 8)), "GCGCAU"), rand_seq(rng, int(rng.integers(4, 8)), "GCGCAU")))
    for k, (s1, s2) in enumerate(cases):
        n1, n2 = len(s1), len(s2)
        allow = None
        if k % 3 == 1:
            m, bp, unp = problem_view(*random_constraint(rng, n1, n2), n1, n2, 2)
            allow = allowed_matrix(m, bp, unp)
        E = random_energies(rng, n1 + n2) if k % 4 >= 2 else None
        U = random_energies(rng, n1 + n2, 150) if k % 2 else None
        assert morc(s1 + s2, n1 + 1, allow, E, U) == _brute(model, s1 + s2, n1 + 1, allow, E, U), (s1, s2, k)


def test_oracle_joined_structures_pay_duplex_init(morc, model):
    """MFE_co = min(MFE_s1 + MFE_s2, joined + DuplexInit) when nothing else differs"""
    s1, s2 = "GGGGAAACCCC", "GGGGAAACCCC"
    co = morc(s1 + s2, len(s1) + 1)
    assert co <= morc(s1) + morc(s2)
    import copy
    m = copy.deepcopy(model)
    m.DuplexInit37 = 100000
    assert morc(s1 + s2, len(s1) + 1, m=m) == morc(s1) + morc(s2)


# ---------------------------------------------------------------------------------------- emulator (CPU)
def _keys_of(m, bp, unp):
    """keys with the library's rule (pair allowed iff equal keys): brute-force from the allowed matrix is not needed --
    the emulator takes any key vector, and this one reproduces allowed_matrix"""
    partner = {}
    for p, q in bp:
        partner[p], partner[q] = q, p
    key = [0] * (m + 1)
    opened, count = [], 0
    for i in range(1, m + 1):
        if i in unp:
            key[i] = 0x8000 + i
        elif i in partner and partner[i] > i:
            count += 1
            opened.append(count)
            key[i] = 2 * count + 1
        elif i in partner:
            key[i] = key[partner[i]]
            opened.pop()
        else:
            key[i] = 2 * opened[-1] if opened else 0
    return np.array(key[1:], dtype=np.uint16)


def _emul_cases(rng, bundled):
    seqs = bundled["sequences"]
    out = [(seqs["DIS"], "", None), (seqs["DIS"], seqs["DIS"], None)]
    for n1, n2 in ((37, 0), (60, 0), (120, 0), (210, 0), (23, 31), (70, 45), (130, 90)):
        out.append((rand_seq(rng, n1), rand_seq(rng, n2), True))
    return out


@pytest.mark.parametrize("T", [32, 64, 160])
def test_emulator_equals_oracle(kemul, morc, model, bundled, T):
    rng = np.random.default_rng(410 + T)
    for k, (s1, s2, data) in enumerate(_emul_cases(rng, bundled)):
        n1, n2 = len(s1), len(s2)
        seq, cp, n = s1 + s2, (n1 + 1 if n2 else 0), n1 + n2
        for variant in range(4 if data else 1):
            keys = allow = E = U = None
            if variant & 1:
                c1, c2 = random_constraint(rng, n1, n2)
                m, bp, unp = problem_view(c1, c2 if n2 else None, n1, n2, 2 if n2 else 0)
                allow = allowed_matrix(m, bp, unp)
                keys = _keys_of(m, bp, unp)
            if variant >= 2:
                E = random_energies(rng, n)
                U = random_energies(rng, n, 150) if variant == 3 else None
            want = morc(seq, cp, allow, E, U)
            lock = n <= 80
            pt, e = emul(kemul, model, seq, cp, keys, E, U, lockstep=False, T=T)
            assert e == want, (k, variant)
            check_structure(model, seq, cp, pt, e, allow, E, U)
            if lock:
                pt2, e2 = emul(kemul, model, seq, cp, keys, E, U, lockstep=True, T=T)
                assert e2 == want and np.array_equal(pt, pt2), (k, variant)


def test_emulator_bundled_pairs(kemul, morc, model, bundled):
    seqs = bundled["sequences"]
    for a, b in bundled["pairs"][:3]:
        s1, s2 = seqs[a], seqs[b]
        for seq, cp in ((s1, 0), (s1 + s2, len(s1) + 1)):
            pt, e = emul(kemul, model, seq, cp, T=256)
            assert e == morc(seq, cp)
            check_structure(model, seq, cp, pt, e)


# ------------------------------------------------------------------------------------- planning and errors (CPU)
def run_shim(shim, pairs, cons=None, stack=None, unpaired=None, problems=7, facts=(148, 1, 0, 180 << 30)):
    keep = []
    n = len(pairs)
    arr = (RpPair * max(n, 1))()
    carr = (RpConstraint * max(n, 1))() if cons else None
    sarr = (RpStackEnergy * max(n, 1))() if stack else None
    uarr = (RpUnpairedEnergy * max(n, 1))() if unpaired else None
    for k, (s1, s2) in enumerate(pairs):
        b = [s1.encode(), s2.encode()]
        keep.append(b)
        arr[k].s1, arr[k].n1, arr[k].s2, arr[k].n2 = b[0], len(s1), (b[1] or None), len(s2)
        if cons and cons[k]:
            c = [x.encode() if x is not None else None for x in cons[k]]
            keep.append(c)
            carr[k].c1, carr[k].c2 = c
        for vec, st, f in ((stack, sarr, "e"), (unpaired, uarr, "u")):
            if vec and vec[k]:
                for s, v in enumerate(vec[k]):
                    if v is not None:
                        a = np.ascontiguousarray(v, dtype=np.float64)
                        keep.append(a)
                        setattr(st[k], f"{f}{s + 1}", a.ctypes.data)
    fa = np.array(facts, dtype=np.int64)
    msg = C.create_string_buffer(400)
    lay = np.zeros((max(n, 1), 6), dtype=np.int64)
    jobs = np.zeros((3 * max(n, 1), 8), dtype=np.int64)
    scal = np.zeros(5, dtype=np.int64)
    cap = sum(2 * (len(a) + len(b)) + 4 for a, b in pairs) + 16
    es, eu, key = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.uint16)
    rc = shim.mfe_shim(arr, carr, sarr, uarr, n, problems, fa.ctypes.data, msg, 400, lay.ctypes.data, jobs.ctypes.data,
                       3 * max(n, 1), scal.ctypes.data, es.ctypes.data, eu.ctypes.data, key.ctypes.data, cap)
    return rc, msg.value.decode(), lay[:n], jobs[:int(scal[1])], scal, es, eu, key


def test_plan_layout_is_the_sample_layout(lib, shim):
    from ractip_b200.stage import sample_opts
    from ractip_b200._lib import RpSampleLayout
    pairs = [("ACGU" * 10, "GGGAAACCC"), ("GGGGAAAACCCC", ""), ("A" * 5, "C" * 7)]
    for problems in range(8):
        rc, msg, lay, jobs, scal, *_ = run_shim(shim, pairs, problems=problems)
        assert rc == 0, msg
        arr = (RpPair * 3)()
        keep = [(a.encode(), b.encode()) for a, b in pairs]
        for k, (a, b) in enumerate(keep):
            arr[k].s1, arr[k].n1, arr[k].s2, arr[k].n2 = a, len(a), b or None, len(b)
        so = sample_opts(1, 1, [nm for nm, bit in (("s1", 1), ("s2", 2), ("co", 4)) if problems & bit])
        want = (RpSampleLayout * 3)()
        tot = C.c_size_t()
        assert lib.rp_sample_plan(arr, 3, C.byref(so), want, C.byref(tot)) == 0
        assert scal[0] == tot.value
        for k in range(3):
            w = want[k]
            assert lay[k].tolist() == [w.s1, w.s2, w.co, w.len_s1, w.len_s2, w.len_co]
        # one job per problem with room, longest first; the lone s1 has no s2 and no co-fold
        assert len(jobs) == sum(1 for k in range(3) for x in lay[k][3:] if x)
        assert list(jobs[:, 1]) == sorted(jobs[:, 1], reverse=True)


def test_plan_rounding_flags_and_constants(shim):
    pairs = [("GGGAAACCCUU", "ACGUACGU")]
    u1 = np.array([0.005, -0.005, 0.0049999, 0.015, -0.025, 1.234, 0, 0, 0, 0, 0])
    e2 = np.array([0.3, 0, 0, 0, 0, 0, 0, -0.2])
    rc, msg, lay, jobs, scal, es, eu, key = run_shim(shim, pairs, cons=[("x..........", None)], stack=[(None, e2)],
                                                     unpaired=[(u1, None)])
    assert rc == 0, msg
    by = {int(j[5]) % 3: j for j in jobs}
    assert by[0][3] == CON_KEYS | CON_UNPAIRED and by[1][3] == CON_STACK
    assert by[2][3] == CON_KEYS | CON_STACK | CON_UNPAIRED
    assert by[0][6] == dcal(u1).sum() == 1 - 1 + 0 + 2 - 3 + 123 and by[1][6] == 0 and by[2][6] == by[0][6]
    off1, off12 = int(by[0][0]), int(by[2][0])
    np.testing.assert_array_equal(eu[off1:off1 + 11], dcal(u1))
    np.testing.assert_array_equal(eu[off12:off12 + 11], dcal(u1))
    np.testing.assert_array_equal(es[int(by[1][0]):int(by[1][0]) + 8], dcal(e2))
    np.testing.assert_array_equal(es[off12 + 11:off12 + 19], dcal(e2))
    assert key[off1] != 0 and key[off12] != key[off12 + 5]   # 'x': unpaired in s1 and in the co-fold


def test_plan_overflow_bound_both_sides(shim):
    n = 500
    s = "GGGAAACCCA" * 50
    lim = RP_INF // 4                     # sum |E| in 0.01 kcal/mol
    u = np.full(n, lim // n / 100.0)      # exactly at the bound
    u[0] += (lim - (lim // n) * n) / 100.0
    assert dcal(u).sum() == lim
    assert run_shim(shim, [(s, "")], unpaired=[(u, None)])[0] == 0
    u2 = u.copy()
    u2[1] += 0.01
    rc, msg, *_ = run_shim(shim, [(s, "")], unpaired=[(u2, None)])
    assert rc == RP_ERR_UNSUPPORTED and msg.startswith("pair 0, problem s1: the pseudo-energies give sum |E| = 25000.01"), msg
    # the co-fold adds both strands (stacking and unpaired), s1 and s2 alone stay inside
    half = np.full(n, lim / 2 / n / 100.0)
    rc, msg, *_ = run_shim(shim, [(s, s)], stack=[(half, None)], unpaired=[(None, half + 0.01)])
    assert rc == RP_ERR_UNSUPPORTED and msg.startswith("pair 0, problem s1&s2:"), msg
    assert run_shim(shim, [(s, s)], stack=[(half, None)], unpaired=[(None, half + 0.01)], problems=3)[0] == 0
    # huge values are rejected, not converted
    rc, msg, *_ = run_shim(shim, [(s, "")], stack=[(np.full(n, 1e300), None)])
    assert rc == RP_ERR_UNSUPPORTED


def test_plan_errors_match_the_probed_batch(shim):
    """the messages of check_constraints, check_stack_energies and check_unpaired_energies (test_unpaired.py,
    test_shape.py, test_constraints.py pin the same texts for the probed batch)"""
    pairs = [("ACGU" * 5, "ACGU"), ("GGGAAACCC", "GGGU")]
    assert run_shim(shim, pairs, problems=8)[:2] == (RP_ERR_ARG, "unknown bits 0x8 in the requested problems")
    bad = np.zeros(4)
    bad[2] = float("nan")
    assert run_shim(shim, pairs, unpaired=[None, (None, bad)])[:2] == (RP_ERR_ARG, "pair 1, u2, position 3: nan kcal/mol is not finite")
    assert run_shim(shim, pairs, stack=[None, (None, bad)])[:2] == (RP_ERR_ARG, "pair 1, e2, position 3: nan kcal/mol is not finite")
    rc, msg, *_ = run_shim(shim, pairs, cons=[None, ("((....)..", None)])
    assert rc == RP_ERR_ARG and msg.startswith("pair 1, c1, position")
    # the pf_scale range of the probed batch does not apply: B = 500 * 300 * 10 / kT = 2433 >> ln 10^150
    big = np.full(500, 3.0)
    assert run_shim(shim, [("GGGAAACCCA" * 50, "")], unpaired=[(big, None)])[0] == 0


def test_plan_memory_budget(shim):
    pairs = [("GGGAAACCC" * 100, "")] * 40
    rc, msg, lay, jobs, scal, *_ = run_shim(shim, pairs, problems=1, facts=(148, 1, 0, 1 << 30))
    assert rc == 0 and scal[2] >= 1
    slot = int(scal[3]) * 4
    assert scal[2] * slot <= (1 << 30) // 10 * 7 or scal[2] == 1
    rc, msg, lay, jobs, scal, *_ = run_shim(shim, pairs, problems=1)
    assert scal[2] == 40


# ----------------------------------------------------------------------------------------- front end (CPU)
def test_format_result_mfe_lines():
    from ractip_b200.frontend import FastaRecord, PairResult, format_result
    from ractip_b200.ip import JointPrediction
    a, b = FastaRecord("a", "GGGAAAACCC"), FastaRecord("b", "GGGUUUCCC")
    j = JointPrediction("..........", ".........", None, None, None)
    t1 = np.array([10, 9, 0, 0, 0, 0, 0, 0, 2, 1], dtype=np.int16)
    t2 = np.zeros(9, dtype=np.int16)
    co = np.zeros(19, dtype=np.int16)
    co[0], co[18] = 19, 1
    r = PairResult(a, b, j, samples=[("[.........", "........]")],
                   mfe={"s1": (t1, -1.5), "s2": (t2, 0.0), "co": (co, -12.345)})
    lines = format_result(r).split("\n")
    assert lines[-4] == "[.........&........]"
    assert lines[-3:] == ["MFE s1: ((......)) (-1.50)", "MFE s2: ......... (0.00)",
                          "MFE s1&s2: [.........&........] (-12.35)"]
    r.mfe = None
    assert "MFE" not in format_result(r)


# --------------------------------------------------------------------------------------------------- GPU
def _stage(model):
    from ractip_b200 import ProbabilityStage
    return ProbabilityStage(model)


@gpu
def test_gpu_bundled_pairs_equal_the_oracle(morc, model, bundled, kemul):
    seqs = bundled["sequences"]
    pairs = [(seqs["DIS"], seqs["DIS"])] + [(seqs[a], seqs[b]) for a, b in bundled["pairs"]]
    st = _stage(model)
    try:
        res = st.mfe(pairs)
    finally:
        st.close()
    for (s1, s2), r in zip(pairs, res):
        for name, seq, cp in (("s1", s1, 0), ("s2", s2, 0), ("co", s1 + s2, len(s1) + 1)):
            t, e = r[name]
            want = morc(seq, cp)
            assert round(e * 100) == want, (name, len(s1), len(s2))
            check_structure(model, seq, cp, t, want)
            if len(seq) <= 400:
                pt, ee = emul(kemul, model, seq, cp, T=512)
                assert ee == want and np.array_equal(pt, t), name


def _random_data(rng, pairs, kind):
    """constraints / stacking / unpaired pseudo-energies of kind bits 1 / 2 / 4"""
    cons = [random_constraint(rng, len(a), len(b)) for a, b in pairs] if kind & 1 else None
    st = [(dcal_inv(random_energies(rng, len(a))), dcal_inv(random_energies(rng, len(b)))) for a, b in pairs] if kind & 2 else None
    un = [(dcal_inv(random_energies(rng, len(a), 150)), dcal_inv(random_energies(rng, len(b), 150)))
          for a, b in pairs] if kind & 4 else None
    return cons, st, un


def dcal_inv(E):
    return np.asarray(E, dtype=np.float64) / 100.0


def _oracle_pair(morc, s1, s2, c, st, un):
    n1, n2 = len(s1), len(s2)
    out = {}
    for w, (name, seq, cp) in enumerate((("s1", s1, 0), ("s2", s2, 0), ("co", s1 + s2, n1 + 1))):
        allow = None
        if c is not None:
            m, bp, unp = problem_view(c[0], c[1], n1, n2, w)
            allow = allowed_matrix(m, bp, unp) if m <= 700 else None
            assert allow is not None
        pick = lambda v: None if v is None else (dcal(v[0]) if w == 0 else dcal(v[1]) if w == 1 else
                                                 np.concatenate([dcal(v[0]), dcal(v[1])]))
        out[name] = (seq, cp, allow, pick(st), pick(un))
    return out


@gpu
@pytest.mark.parametrize("kind", [0, 1, 2, 4, 3, 5, 6, 7])
def test_gpu_random_pairs_with_data(morc, model, kemul, kind):
    rng = np.random.default_rng(430 + kind)
    pairs = [(rand_seq(rng, 40), rand_seq(rng, 25)), (rand_seq(rng, 150), rand_seq(rng, 90)),
             (rand_seq(rng, 260), rand_seq(rng, 230)), (rand_seq(rng, 30), "")]
    cons, st, un = _random_data(rng, pairs, kind)
    stage = _stage(model)
    try:
        res = stage.mfe(pairs, cons, st, un)
    finally:
        stage.close()
    for k, ((s1, s2), r) in enumerate(zip(pairs, res)):
        o = _oracle_pair(morc, s1, s2, cons[k] if cons else None, st[k] if st else None, un[k] if un else None)
        for name in ("s1", "s2", "co") if s2 else ("s1",):
            seq, cp, allow, E, U = o[name]
            t, e = r[name]
            want = morc(seq, cp, allow, E, U)
            assert round(e * 100) == want, (k, name)
            check_structure(model, seq, cp, t, want, allow, E, U)
            if len(seq) <= 300:
                key = None
                if allow is not None:
                    m, bp, unp = problem_view(cons[k][0], cons[k][1], len(s1), len(s2), ("s1", "s2", "co").index(name))
                    key = _keys_of(m, bp, unp)
                pt, ee = emul(kemul, model, seq, cp, key, E, U, T=512)
                assert ee == want and np.array_equal(pt, t), (k, name)
        if not s2:
            assert set(r) == {"s1"}


@gpu
def test_gpu_long_cofold(morc, model):
    rng = np.random.default_rng(440)
    s1, s2 = rand_seq(rng, 1000), rand_seq(rng, 500)
    stage = _stage(model)
    try:
        r = stage.mfe([(s1, s2)], problems=("co",))[0]
    finally:
        stage.close()
    t, e = r["co"]
    want = morc(s1 + s2, 1001)
    assert round(e * 100) == want
    check_structure(model, s1 + s2, 1001, t, want)


@gpu
def test_gpu_bounds_against_the_partition_function_and_samples(model0, bundled):
    """-E_mfe/kT <= log Z for every problem (model0: pf_smooth = 0); every sampled structure has E >= MFE"""
    from ractip_b200 import ProbabilityStage, energy_of_structure
    seqs = bundled["sequences"]
    rng = np.random.default_rng(450)
    pairs = [(seqs[a], seqs[b]) for a, b in bundled["pairs"][:4]] + [(rand_seq(rng, 120), rand_seq(rng, 80))]
    st = ProbabilityStage(model0)
    try:
        mf = st.mfe(pairs)
        b = st.batch(pairs, samples=20, sample_seed=3)
        try:
            b.run()
            logz = b.fetch_logz()
            smp = b.fetch_samples()
        finally:
            b.close()
        alone = [st.mfe([p])[0] for p in pairs[::2]]
    finally:
        st.close()
    kt = KT / 1000.0
    for k, ((s1, s2), r) in enumerate(zip(pairs, mf)):
        for w, (name, seq, cp) in enumerate((("s1", s1, -1), ("s2", s2, -1), ("co", s1 + s2, len(s1) + 1))):
            t, e = r[name]
            # the partition function leaves DuplexInit out: compare without it for a joined MFE structure
            joined = cp > 0 and any(i < cp <= j for i, j in pairs_of(t))
            e_pf = e - (model0.DuplexInit37 / 100.0 if joined else 0.0)
            assert -e_pf / kt <= logz[k][w] + 1e-6, (k, name)
            for tt in smp[k][name]:
                es = energy_of_structure(model0, seq, dot_bracket_str(tt), cp)
                assert round(es * 100) >= round(e * 100), (k, name)
    for r, a in zip(mf[::2], alone):   # a pair's MFE does not depend on the other pairs of its batch
        for name in r:
            assert r[name][1] == a[name][1] and np.array_equal(r[name][0], a[name][0])


def dot_bracket_str(t):
    from ractip_b200 import dot_bracket
    return dot_bracket(t)


@gpu
def test_gpu_command_line(bundled, tmp_path):
    seqs = bundled["sequences"]
    a, b = bundled["pairs"][0]
    s1, s2 = seqs[a], seqs[b]
    fa1, fa2 = tmp_path / "a.fa", tmp_path / "b.fa"
    fa1.write_text(f">a\n{s1}\n" + "." * len(s1) + "\n")
    fa2.write_text(f">b\n{s2}\n" + "x" + "." * (len(s2) - 1) + "\n")
    shp = tmp_path / "a.shape"
    shp.write_text("".join(f"{i} {0.1 * (i % 7)}\n" for i in range(1, len(s1) + 1)))
    run = lambda *args: subprocess.run([sys.executable, "-m", "ractip_b200", str(fa1), str(fa2), *args], cwd=ROOT,
                                       capture_output=True, text=True)
    for extra in ([], ["-c"], ["--shape", f"a={shp}"], ["--shape", f"a={shp}", "--shape-method", "W", "-c"],
                  ["--sample", "2"]):
        base, with_mfe = run(*extra), run(*extra, "--mfe")
        assert base.returncode == 0 and with_mfe.returncode == 0, with_mfe.stdout + with_mfe.stderr
        lines = with_mfe.stdout.rstrip("\n").split("\n")
        assert "\n".join(lines[:-3]) == base.stdout.rstrip("\n")
        assert lines[-3].startswith("MFE s1: ") and lines[-2].startswith("MFE s2: ") and lines[-1].startswith("MFE s1&s2: ")
        r1, r2 = lines[-1].split(" ")[2].split("&")
        assert len(r1) == len(s1) and len(r2) == len(s2)
        if "-c" in extra:
            assert r2[0] == "." and lines[-2].split(" ")[2][0] == "."
