"""Stochastic sampling of secondary structures: the sampling phase of the general kernel (mcc_sample.h).

The oracle sampler (tests/cpp/oracle_sample.c) draws on the soft oracle's tables with the same Philox numbers, decision
order and selection rule; it is pinned by exhaustive enumeration of every structure's exact probability.  CPU: Philox
against numpy and a known answer, the oracle sampler against enumeration, the kernel's sampling phase in the host
emulator against the oracle sampler sample by sample, planning, errors, helpers and the command line.  GPU: the
library against the oracle sampler sample by sample and against enumeration, marginals, byte identity of everything
that is not sampled, tensors and the command line."""
import ctypes as C
import math
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from ractip_b200._lib import RpConstraint, RpOpts, RpPair, RpSampleLayout, RpSampleOpts, RpStackEnergy

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(Path(__file__).resolve().parent))
from conftest import rand_seq  # noqa: E402
from test_constraints import allowed_matrix, problem_view, random_constraint  # noqa: E402
from test_ip import all_structures, can_pair, to_string  # noqa: E402

RP_ERR_ARG, RP_ERR_CAPACITY, RP_ERR_UNSUPPORTED = 1, 9, 10
CON_KEYS, CON_STACK, CON_SAMPLE = 1, 2, 4
KT = (37.0 + 273.15) * 1.98717   # cal/mol
TOL = 2e-7
ROUTES = [(0, 1), (5, 1), (10, 1), (15, 1), (10, 8), (10, 16)]
ROUTE_ENVS = [{}, {"RP_MCC_LONG_N": "1", "RP_CLUSTER": "0"}, {"RP_CLUSTER": "8"}, {"RP_CLUSTER": "16"}]
gpu = pytest.mark.gpu


def _cc(cmd):
    subprocess.run(cmd, check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)


def random_energies(rng, n):
    """integer pseudo-energies (0.01 kcal/mol): many zeros, negatives, a few large ones"""
    E = rng.integers(-300, 300, size=n)
    E[rng.random(n) < 0.3] = 0
    big = rng.random(n) < 0.08
    E[big] = rng.choice([-900, 1500, 4000], size=int(big.sum()))
    return E.astype(np.int32)


def opts(**kw):
    o = dict(max_w=15, min_w=5, th_ss=0.5, th_hy=0.1, th_ac=0.003, use_pf_duplex=0)
    o.update(kw)
    return RpOpts(**o)


# ------------------------------------------------------------------------------------------------ oracle sampler
class SampleOracle:
    def __init__(self, so, model):
        self.lib = C.CDLL(str(so))
        vp, i = C.c_void_p, C.c_int
        self.lib.orc_params_new.restype = vp
        self.lib.orc_params_new.argtypes = [vp]
        self.lib.orc_fold_soft.restype = i
        self.lib.orc_fold_soft.argtypes = [vp, C.c_char_p, i, i, vp, vp, vp, vp, i, vp]
        self.lib.orc_sample_soft.restype = i
        self.lib.orc_sample_soft.argtypes = [vp, C.c_char_p, i, i, vp, vp, C.c_uint64, i, i, i, i, vp]
        self.lib.orc_philox.argtypes = [vp, vp, vp]
        self._model = model
        self.P = self.lib.orc_params_new(C.addressof(model))

    @staticmethod
    def _arrs(allow, E):
        a = None if allow is None else np.ascontiguousarray(allow, dtype=np.uint8)
        e = None if E is None else np.ascontiguousarray(E, dtype=np.int32)
        return a, e, (None if a is None else a.ctypes.data), (None if e is None else e.ctypes.data)

    def fold(self, seq, cp=0, allow=None, E=None, max_w=0):
        n = len(seq)
        pr, up, lz = np.zeros((n + 1, n + 1)), np.zeros((n, max(max_w, 1))), C.c_double()
        a, e, pa, pe = self._arrs(allow, E)
        assert self.lib.orc_fold_soft(self.P, seq.encode(), n, cp, pa, pe, pr.ctypes.data, up.ctypes.data, max_w,
                                      C.byref(lz)) == 0
        return pr, up, lz.value

    def sample(self, seq, cp=0, allow=None, E=None, seed=1, pair=0, kind=0, num=1, first=0):
        n = len(seq)
        out = np.zeros((num, n), dtype=np.int16)
        a, e, pa, pe = self._arrs(allow, E)
        assert self.lib.orc_sample_soft(self.P, seq.encode(), n, cp, pa, pe, seed, pair, kind, first, num,
                                        out.ctypes.data) == 0
        return out

    def philox(self, ctr, key):
        c = np.array(ctr, dtype=np.uint64)
        k = np.array(key, dtype=np.uint64)
        out = np.zeros(4, dtype=np.uint64)
        self.lib.orc_philox(c.ctypes.data, k.ctypes.data, out.ctypes.data)
        return [int(x) for x in out]


def _build_oracle(tmp_path_factory):
    so = tmp_path_factory.mktemp("sorc") / "liboracle_sample.so"
    _cc(["gcc", "-O3", "-fPIC", "-shared", "-I", str(ROOT / "include"), "-I", str(ROOT / "ractip_b200" / "csrc"),
         str(ROOT / "tests" / "cpp" / "oracle_sample.c"), "-o", str(so), "-lm"])
    return so


@pytest.fixture(scope="module")
def orc_so(tmp_path_factory, lib):
    return _build_oracle(tmp_path_factory)


@pytest.fixture(scope="module")
def sorc(orc_so, model):
    return SampleOracle(orc_so, model)


@pytest.fixture(scope="module")
def model0(lib):
    """the default model with the clipped tables (pf_smooth = 0) that the integer energy evaluation uses"""
    from ractip_b200 import default_model
    m = default_model()
    m.pf_smooth = 0
    return m


@pytest.fixture(scope="module")
def sorc0(orc_so, model0):
    return SampleOracle(orc_so, model0)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = tmp_path_factory.mktemp("smpshim") / "libsample_shim.so"
    csrc = ROOT / "ractip_b200" / "csrc"
    _cc(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", str(ROOT / "include"), "-I", str(csrc),
         str(csrc / "plan.cpp"), str(ROOT / "tests" / "cpp" / "sample_shim.cpp"), "-o", str(so)])
    lib = C.CDLL(str(so))
    vp = C.c_void_p
    lib.sample_shim.argtypes = [vp, vp, vp, C.c_int, vp, vp, C.c_char_p, C.c_int, vp, vp, C.c_int, vp, vp]
    lib.sample_shim.restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def kemul(tmp_path_factory):
    so = tmp_path_factory.mktemp("smpemul") / "libemul_sampled.so"
    d = ROOT / "tests" / "emul"
    _cc(["g++", "-O2", "-U_FORTIFY_SOURCE", "-std=c++17", "-fPIC", "-shared", "-I", str(ROOT / "ractip_b200" / "csrc"),
         "-I", str(ROOT / "include"), "-o", str(so), str(d / "emul_sampled.cpp"),
         str(ROOT / "ractip_b200" / "csrc" / "dev_model.cpp")])
    lib = C.CDLL(str(so))
    vp, i = C.c_void_p, C.c_int
    lib.emul_sampled_problem.argtypes = [i, i, i, vp, vp, vp, C.c_char_p, i, i, i, i, i, C.c_uint64, i, i, vp, vp]
    lib.emul_sampled_problem.restype = i
    return lib


# ------------------------------------------------------------------------------------------------ Philox (CPU)
def test_philox_known_answer_and_numpy(sorc):
    # Random123's known-answer vectors of Philox4x64-10
    assert sorc.philox([0, 0, 0, 0], [0, 0]) == [0x16554d9eca36314c, 0xdb20fe9d672d0fdc, 0xd7e772cee186176b,
                                                 0x7e68b68aec7ba23b]
    pi_ctr = [0x243f6a8885a308d3, 0x13198a2e03707344, 0xa4093822299f31d0, 0x082efa98ec4e6c89]
    pi_key = [0x452821e638d01377, 0xbe5466cf34e90c6c]
    assert sorc.philox(pi_ctr, pi_key) == [0xa528f45403e61d95, 0x38c72dbd566e9788, 0xa5a1610e72fd18b5,
                                           0x57bd43b5e52b7fe6]
    # numpy.random.Philox increments its counter before each block: the block of counter c is Philox(counter=c-1)'s
    rng = np.random.default_rng(5)
    words = lambda v, k: sum(int(x) << (64 * t) for t, x in enumerate(v[:k]))
    for _ in range(12):
        ctr = [int(x) for x in rng.integers(0, 2 ** 63, 4, dtype=np.uint64)]
        key = [int(x) for x in rng.integers(0, 2 ** 63, 2, dtype=np.uint64)]
        if rng.random() < 0.3:
            ctr[1:] = [0, 0, 0]
        g = np.random.Philox(key=words(key, 2), counter=(words(ctr, 4) - 1) % (1 << 256))
        assert sorc.philox(ctr, key) == [int(x) for x in g.random_raw(4)]


# ------------------------------------------------------------------------ oracle sampler vs enumeration (CPU)
def exact_distribution(model0, sorc0, seq, cp, allow, E):
    """{pair table bytes: probability} of every structure, from the integer energy evaluation: E(S), minus DuplexInit
    for a structure that joins the strands, plus its stacks' pseudo-energies, over the oracle's Z"""
    from ractip_b200 import energy_of_structure
    n = len(seq)
    _, _, logz = sorc0.fold(seq, cp, allow, E, 0)
    kT = KT / 1000.0
    out = {}
    for pairs in all_structures(n):
        if not all(can_pair(seq[i - 1], seq[j - 1]) for i, j in pairs):
            continue
        if allow is not None and not all(allow[i, j] for i, j in pairs):
            continue
        e = energy_of_structure(model0, seq, to_string(n, pairs), cp if cp else -1)
        if cp and any(i < cp <= j for i, j in pairs):
            e -= model0.DuplexInit37 / 100.0
        if E is not None:
            pt = dict(pairs)
            for i, j in pairs:
                if pt.get(i + 1) == j - 1 and not (cp and i < cp <= j):
                    e += (E[i - 1] + E[i] + E[j - 2] + E[j - 1]) / 100.0
        t = np.zeros(n, dtype=np.int16)
        for i, j in pairs:
            t[i - 1], t[j - 1] = j, i
        out[t.tobytes()] = math.exp(-e / kT - logz)
    assert abs(sum(out.values()) - 1.0) < 1e-3   # the evaluation and the DP describe one ensemble
    return out


def check_distribution(tables, exact):
    """every structure with an expected count >= 20 within 6 sigma, nothing outside the ensemble, and a total variation
    distance below three times its expectation bound 0.5 sum_S sqrt(p_S / N)"""
    N = len(tables)
    counts = {}
    for t in tables:
        k = t.tobytes()
        counts[k] = counts.get(k, 0) + 1
    assert set(counts) <= set(exact), "a sample outside the ensemble"
    for k, p in exact.items():
        if N * p >= 20:
            c = counts.get(k, 0)
            assert abs(c - N * p) <= 6 * math.sqrt(N * p * (1 - p)), (c, N * p)
    tvd = 0.5 * sum(abs(counts.get(k, 0) / N - p) for k, p in exact.items())
    bound = 3 * 0.5 * sum(math.sqrt(p / N) for p in exact.values())
    assert tvd < bound, (tvd, bound)


ENUM_CASES = ["plain", "constraint", "energies", "both"]


def enum_inputs(case):
    """the enumeration cases, a 12-nt strand and 7+5 nt with a cut point: dicts of the pair (s1, s2), the oracle's
    inputs (seq, cp, allow, E) and the library's (cons, energies in kcal/mol)"""
    rng = np.random.default_rng(200 + ENUM_CASES.index(case))
    out = []
    for n1, n2 in ((12, 0), (7, 5)):
        s = rand_seq(rng, n1 + n2, "GCGCAU")
        cp = n1 + 1 if n2 else 0
        d = dict(pair=(s[:n1], s[n1:]), seq=s, cp=cp, allow=None, E=None, cons=None, energies=None)
        if case in ("constraint", "both"):
            d["cons"] = random_constraint(rng, n1, n2, 0.2)
            m, bp, unp = problem_view(*d["cons"], n1, n2, 2 if n2 else 0)
            d["allow"] = allowed_matrix(m, bp, unp)
        if case in ("energies", "both"):
            d["E"] = random_energies(rng, n1 + n2)
            d["energies"] = (d["E"][:n1] / 100.0, d["E"][n1:] / 100.0 if n2 else None)
        out.append(d)
    return out


@pytest.mark.parametrize("case", ENUM_CASES)
def test_oracle_sampler_matches_enumeration(model0, sorc0, case):
    for d in enum_inputs(case):
        exact = exact_distribution(model0, sorc0, d["seq"], d["cp"], d["allow"], d["E"])
        tables = sorc0.sample(d["seq"], d["cp"], d["allow"], d["E"], seed=7, pair=3, kind=2 if d["cp"] else 0, num=100000)
        check_distribution(tables, exact)


def test_oracle_sampler_streams(sorc):
    """a sample depends on (seed, pair, kind, index) only: a range drawn alone equals the same rows of a longer run"""
    rng = np.random.default_rng(9)
    s = rand_seq(rng, 60)
    a = sorc.sample(s, 0, None, None, seed=11, pair=2, kind=1, num=40)
    assert np.array_equal(sorc.sample(s, 0, None, None, seed=11, pair=2, kind=1, num=15, first=25), a[25:])
    assert not np.array_equal(sorc.sample(s, 0, None, None, seed=12, pair=2, kind=1, num=40), a)
    assert not np.array_equal(sorc.sample(s, 0, None, None, seed=11, pair=3, kind=1, num=40), a)
    for t in a:   # pair tables: symmetric, nested, hairpins of at least 3
        for i, j in enumerate(t, 1):
            if j:
                assert t[j - 1] == i and abs(j - i) > 3
        st = []
        for i, j in enumerate(t, 1):
            if j > i:
                st.append(j)
            elif j and j < i:
                assert st.pop() == i


# -------------------------------------------------------------------------------------------- planning (CPU)
def plan(shim, pairs, so, cons=None, o=None):
    """(rc, message, key buffer, per-problem (seq_off, n, constrained, general), same plan as without samples)"""
    keep = []
    arr = (RpPair * len(pairs))()
    carr = (RpConstraint * len(pairs))() if cons else None
    for k, (s1, s2) in enumerate(pairs):
        b = [s1.encode(), s2.encode()]
        keep.append(b)
        arr[k].s1, arr[k].n1, arr[k].s2, arr[k].n2 = b[0], len(s1), b[1] or None, len(s2)
        if cons:
            c = [x.encode() if x is not None else None for x in cons[k]]
            keep.append(c)
            carr[k].c1, carr[k].c2 = c
    cap = sum(2 * (len(a) + len(b)) + 4 for a, b in pairs) + 16
    key = np.zeros(cap, dtype=np.uint16)
    klen = C.c_longlong()
    probs = np.zeros((3 * len(pairs), 4), dtype=np.int64)
    same = C.c_int()
    msg = C.create_string_buffer(256)
    o = o or opts()
    rc = shim.sample_shim(arr, carr, None, len(pairs), C.byref(o), C.byref(so) if so is not None else None, msg, 256,
                          key.ctypes.data, C.byref(klen), cap, probs.ctypes.data, C.byref(same))
    return rc, msg.value.decode(), key[:klen.value], probs, bool(same.value)


def test_routing(shim):
    rng = np.random.default_rng(31)
    pairs = [(rand_seq(rng, 90), rand_seq(rng, 70)), (rand_seq(rng, 40), ""), (rand_seq(rng, 120), rand_seq(rng, 60))]
    rc, _, _, base, same = plan(shim, pairs, None)
    assert rc == 0 and same and not base[:, 2].any() and not base[:, 3][base[:, 1] > 0].all()
    for num, probs_ in ((0, ("s1", "s2", "co")), (5, ("s2",)), (5, ("s1", "co")), (3, ("s1", "s2", "co"))):
        from ractip_b200 import sample_opts
        so = sample_opts(num, 1, probs_)
        rc, _, _, pr, same = plan(shim, pairs, so)
        assert rc == 0
        assert same == (num == 0)
        for k in range(len(pairs)):
            for which, name in enumerate(("s1", "s2", "co")):
                row = pr[3 * k + which]
                want = num > 0 and name in probs_ and row[1] > 0
                assert bool(row[2] & CON_SAMPLE) == want, (k, name)
                if want:
                    assert row[3] == 1   # on the general kernel
                else:
                    assert row[2] == 0 and row[3] == base[3 * k + which][3]   # keeps its route


def test_sample_plan(lib):
    from ractip_b200 import sample_opts
    pairs = [("ACGU" * 5, "GGCC" * 3), ("ACG" * 7, ""), ("A" * 9, "U" * 4)]
    keep = [(a.encode(), b.encode()) for a, b in pairs]
    arr = (RpPair * 3)()
    for k, (a, b) in enumerate(keep):
        arr[k].s1, arr[k].n1, arr[k].s2, arr[k].n2 = a, len(a), b or None, len(b)
    lay = (RpSampleLayout * 3)()
    tot = C.c_size_t()
    so = sample_opts(7, 3, ("s1", "co"))
    assert lib.rp_sample_plan(arr, 3, C.byref(so), lay, C.byref(tot)) == 0
    off = 0
    for k, (a, b) in enumerate(pairs):
        L = lay[k]
        want = [(7 * len(a)), 0, 7 * (len(a) + len(b)) if b else 0]
        assert [L.len_s1, L.len_s2, L.len_co] == want
        assert [L.s1, L.s2, L.co] == [off, off + want[0], off + want[0] + want[1]]
        off += sum(want)
    assert tot.value == off
    assert lib.rp_sample_plan(arr, 3, C.byref(RpSampleOpts(-1, 1, 7)), lay, C.byref(tot)) == RP_ERR_ARG
    assert lib.rp_sample_plan(arr, 3, None, lay, C.byref(tot)) == RP_ERR_ARG
    # an overflow of the running offset
    many = (RpPair * 4)()
    for k in range(4):
        many[k].s1, many[k].n1, many[k].s2, many[k].n2 = b"A", 2 ** 31 - 1, b"A", 2 ** 31 - 1
    lay4 = (RpSampleLayout * 4)()
    assert lib.rp_sample_plan(many, 4, C.byref(RpSampleOpts(2 ** 31 - 1, 1, 7)), lay4, C.byref(tot)) == RP_ERR_ARG


def test_bad_options(shim):
    pairs = [("GGGAAACCC", "GGGUUUCCC"), ("GGGGAAAACCCC", "")]
    for so, code, msg in ((RpSampleOpts(-2, 1, 7), RP_ERR_ARG, "sample count -2 is negative"),
                          (RpSampleOpts(3, 1, 9), RP_ERR_ARG, "unknown bits 0x8 in the sampled problems")):
        rc, m, _, _, _ = plan(shim, pairs, so)
        assert (rc, m) == (code, msg)
    rc, m, _, _, _ = plan(shim, pairs, RpSampleOpts(3, 1, 4), o=opts(use_pf_duplex=1))
    assert (rc, m) == (RP_ERR_UNSUPPORTED, "pair 0: --duplex has no co-fold ensemble to sample")
    rc, _, _, pr, _ = plan(shim, pairs, RpSampleOpts(3, 1, 3), o=opts(use_pf_duplex=1))
    assert rc == 0 and pr[0][2] == CON_SAMPLE and pr[2][2] == 0   # the folds of a --duplex batch can be sampled


# -------------------------------------------------------------------------------------------- helpers (CPU)
def test_joint_structure_is_a_constraint_line(shim, sorc):
    from ractip_b200 import dot_bracket, joint_structure
    rng = np.random.default_rng(41)
    s1, s2 = rand_seq(rng, 30, "GCGCAU"), rand_seq(rng, 25, "GCGCAU")
    n1, n2 = len(s1), len(s2)
    tables = sorc.sample(s1 + s2, n1 + 1, None, None, seed=3, pair=0, kind=2, num=300)
    joined = 0
    for t in tables:
        r1, r2 = joint_structure(t, n1)
        rc, msg, _, _, _ = plan(shim, [(s1, s2)], None, cons=[(r1, r2)])
        assert rc == 0, msg
        # every pair of the sample is allowed in the problem that sees its kind of bracket
        A = [allowed_matrix(*problem_view(r1, r2, n1, n2, w)) for w in range(3)]
        for i, j in enumerate(t, 1):
            if j > i:
                if j <= n1:
                    assert A[0][i, j]
                elif i > n1:
                    assert A[1][i - n1, j - n1]
                else:
                    assert A[2][i, j]
                    joined += 1
    assert joined > 0
    assert dot_bracket(np.array([5, 0, 0, 0, 1, 0])) == "(...)."


# ------------------------------------------------------------------------------ emulator vs oracle sampler (CPU)
def _emul_samples(kemul, model, seq, cp, kind, which, keys, f, route, G, lockstep, num, seed=5, pair=1, T=64):
    n = len(seq)
    out = np.zeros((num, n), dtype=np.int16)
    stk = None if f is None else np.ascontiguousarray(np.concatenate([[1.0], f]))
    key = None if keys is None else np.ascontiguousarray(keys, dtype=np.uint16)
    lz = C.c_double()
    rc = kemul.emul_sampled_problem(route, G, int(lockstep), None if stk is None else stk.ctypes.data,
                                    None if key is None else key.ctypes.data, C.addressof(model), seq.encode(), n, cp,
                                    kind, pair, which, seed, num, T, out.ctypes.data, C.byref(lz))
    assert rc == 0, rc
    return out


@pytest.mark.parametrize("lockstep", [False, True])
def test_emulator_matches_oracle_sample_by_sample(shim, kemul, sorc, model, lockstep):
    rng = np.random.default_rng(71)
    s1, s2 = rand_seq(rng, 47), rand_seq(rng, 38)
    c1, c2 = random_constraint(rng, 47, 38)
    E1, E2 = random_energies(rng, 47), random_energies(rng, 38)
    _, _, keybuf, probs, _ = plan(shim, [(s1, s2)], RpSampleOpts(1, 1, 7), cons=[(c1, c2)])
    num = 24
    for with_data in (False, True):
        for which, seq, cp, kind in ((0, s1, 0, 0), (2, s1 + s2, 48, 1)):
            n = len(seq)
            E = np.concatenate([E1, E2])[:n] if with_data else None
            f = None if E is None else np.exp(-E * 10.0 / KT)
            keys = allow = None
            if with_data:
                off = int(probs[which][0])
                keys = np.concatenate([[0], keybuf[off:off + n]])   # key[1..n]
                m, bp, unp = problem_view(c1, c2, 47, 38, which)
                allow = allowed_matrix(m, bp, unp)
            want = sorc.sample(seq, cp, allow, E, seed=5, pair=1, kind=which, num=num)
            for route, G in ROUTES:
                got = _emul_samples(kemul, model, seq, cp, kind, which, keys, f, route, G, lockstep, num)
                bad = [s for s in range(num) if not np.array_equal(got[s], want[s])]
                assert not bad, (route, G, with_data, which, bad[:3])


# ----------------------------------------------------------------------------------------- front end (CPU)
def _cli(args, cwd=ROOT):
    return subprocess.run([sys.executable, "-m", "ractip_b200"] + args, cwd=cwd, stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True, timeout=900)


def test_command_line_input_errors(tmp_path, lib, bundled):
    seqs = bundled["sequences"]
    (tmp_path / "a.fa").write_text(f">MicA\n{seqs['MicA']}\n")
    (tmp_path / "b.fa").write_text(f">ompA\n{seqs['ompA']}\n")
    fa = [str(tmp_path / "a.fa"), str(tmp_path / "b.fa")]
    for extra, msg in ((["--sample", "3", "--duplex"], "--sample: --duplex has no co-fold ensemble to sample"),
                       (["--sample", "-1"], "--sample -1: the number of samples cannot be negative")):
        r = _cli(extra + fa)
        assert r.returncode == 1 and msg in r.stdout, r.stdout


def test_predict_samples_the_pairs_only(monkeypatch):
    """predict(samples=) draws co-fold samples in the pairs' batch, with constraints and energies, and leaves the
    z-score shuffles unsampled"""
    from types import SimpleNamespace
    from ractip_b200 import frontend
    from ractip_b200.frontend import FastaRecord, format_result
    calls = []

    class FakeBatch:
        def __init__(self, seqs, kw):
            self.seqs = seqs
            calls.append(("batch", seqs, kw))

        def run(self):
            pass

        def fetch_dense(self):
            return None

        def split_dense(self, flat):
            return [SimpleNamespace(bp1=None, bp2=None) for _ in self.seqs]

        def fetch_samples(self):
            t = np.zeros((2, 18), dtype=np.int16)
            t[0, 0], t[0, 17] = 18, 1
            return [{"co": t}]

        def close(self):
            pass

    class FakeStage:
        model = None

        def batch(self, seqs, opts, cons, energies, **kw):
            return FakeBatch(seqs, dict(kw, cons=cons, energies=energies))

        def run_dense(self, seqs, opts, constraints=None, **kw):
            calls.append(("dense", list(seqs), kw))
            return [SimpleNamespace(bp1=None, bp2=None) for _ in seqs]

    monkeypatch.setattr(frontend, "solve_joint", lambda *a, **k: SimpleNamespace(r1="." * 9, r2="." * 9, e1=0.0, e2=0.0, e3=0.0))
    monkeypatch.setattr(frontend, "solve_ss", lambda *a, **k: (None, None, 0.0))
    monkeypatch.setattr(frontend, "zscore_statistic", lambda *a, **k: (0.0, 0.0))
    a, b = FastaRecord("a", "GGGAAACCC"), FastaRecord("b", "GGGUUUCCC")
    res = frontend.predict(FakeStage(), [(a, b)], zscore=12, num_shuffling=2, samples=2, sample_seed=9)
    assert calls[0][0] == "batch" and calls[0][2]["samples"] == 2 and calls[0][2]["sample_seed"] == 9
    assert calls[0][2]["sample_problems"] == ("co",)
    assert calls[1][0] == "dense" and calls[1][2] == {}   # the shuffles: no samples
    assert res[0].samples == [("[........", "........]"), (".........", ".........")]
    assert format_result(res[0]).splitlines()[-2:] == ["[........&........]", ".........&........."]


# ------------------------------------------------------------------------------------------------- GPU
def _stage_env(monkeypatch, env, model=None):
    from ractip_b200 import ProbabilityStage
    for k in ("RP_BAND", "RP_CLUSTER", "RP_MCC_LONG_N"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    return ProbabilityStage(model=model)


def _problem_inputs(s1, s2, which, cons, energies):
    """(seq, cp, allow, E) of problem `which` as the oracle takes it, from one pair's constraint and kcal/mol energies"""
    n1, n2 = len(s1), len(s2)
    seq, cp = ((s1, 0), (s2, 0), (s1 + s2, n1 + 1))[which]
    allow = E = None
    if cons is not None:
        m, bp, unp = problem_view(cons[0], cons[1], n1, n2, which)
        allow = allowed_matrix(m, bp, unp)
    if energies is not None:
        z = lambda e, n: np.zeros(n, dtype=np.int64) if e is None else \
            (np.sign(e) * np.floor(np.abs(e) * 100.0 + 0.5)).astype(np.int64)
        E1, E2 = z(energies[0], n1), z(energies[1], n2)
        E = (E1, E2, np.concatenate([E1, E2]))[which]
    return seq, cp, allow, E


def _sampled(stage, pairs, o, num, seed=1, cons=None, energies=None, problems=("s1", "s2", "co")):
    b = stage.batch(pairs, o, cons, energies, samples=num, sample_seed=seed, sample_problems=problems)
    try:
        b.run()
        flat = b.fetch_dense()
        return b.fetch_samples(), b.split_dense(flat), b.fetch_logz(), flat.copy()
    finally:
        b.close()


def _bundled_data(bundled):
    from ractip_b200 import shape_deigan
    seqs = bundled["sequences"]
    rng = np.random.default_rng(91)
    pairs = [(seqs[a], seqs[b]) for a, b in bundled["pairs"]]
    energies = []
    cons = []
    for s1, s2 in pairs:
        r = lambda n: np.where(rng.random(n) < 0.15, -999.0, rng.gamma(0.6, 0.8, size=n))
        energies.append((shape_deigan(r(len(s1))), shape_deigan(r(len(s2)))))
        cons.append(random_constraint(rng, len(s1), len(s2), 0.1))
    return pairs, cons, energies


_ORACLE_SAMPLES = {}


def _check_against_oracle(sorc, pairs, smp, num, seed, cons=None, energies=None):
    for k, (s1, s2) in enumerate(pairs):
        for which, name in enumerate(("s1", "s2", "co")):
            if name not in smp[k]:
                continue
            c, e = None if cons is None else cons[k], None if energies is None else energies[k]
            tag = (s1, s2, which, str(c), None if e is None else tuple(np.concatenate([x for x in e if x is not None])),
                   num, seed, k)
            if tag not in _ORACLE_SAMPLES:   # (the long pairs are checked on four routes)
                seq, cp, allow, E = _problem_inputs(s1, s2, which, c, e)
                _ORACLE_SAMPLES[tag] = sorc.sample(seq, cp, allow, E, seed=seed, pair=k, kind=which, num=num)
            want = _ORACLE_SAMPLES[tag]
            got = smp[k][name]
            bad = [s for s in range(num) if not np.array_equal(got[s], want[s])]
            assert not bad, (k, name, bad[:3])


@gpu
@pytest.mark.parametrize("env", [{}, {"RP_BAND": "0"}], ids=["default", "no_band"])
@pytest.mark.parametrize("data", [False, True], ids=["bare", "cons_shape"])
def test_gpu_bundled_pairs_match_oracle(sorc, bundled, monkeypatch, env, data):
    pairs, cons, energies = _bundled_data(bundled)
    if not data:
        cons = energies = None
    stage = _stage_env(monkeypatch, env)
    try:
        smp, _, _, _ = _sampled(stage, pairs, opts(), 40, 17, cons, energies)
    finally:
        stage.close()
    _check_against_oracle(sorc, pairs, smp, 40, 17, cons, energies)


@gpu
@pytest.mark.parametrize("env", ROUTE_ENVS, ids=["default", "wide", "cluster8", "cluster16"])
def test_gpu_long_pair_routes(sorc, monkeypatch, env):
    from ractip_b200 import shape_deigan
    rng = np.random.default_rng(82)
    pairs = [(rand_seq(rng, 620), rand_seq(rng, 300)), (rand_seq(rng, 720), rand_seq(rng, 90))]
    energies = [(shape_deigan(rng.gamma(0.6, 0.8, size=len(a))), shape_deigan(rng.gamma(0.6, 0.8, size=len(b))))
                for a, b in pairs]
    cons = [random_constraint(rng, len(a), len(b), 0.05) for a, b in pairs]
    stage = _stage_env(monkeypatch, env)
    try:
        smp, _, _, _ = _sampled(stage, pairs, opts(), 6, 23, cons, energies)
    finally:
        stage.close()
    _check_against_oracle(sorc, pairs, smp, 6, 23, cons, energies)


@gpu
@pytest.mark.parametrize("case", ENUM_CASES)
def test_gpu_exact_distribution(model0, sorc0, monkeypatch, case):
    """the library's samples of the enumeration cases: s1 of the lone strand, the co-fold of the two-strand pair"""
    lone, two = enum_inputs(case)
    pairs = [lone["pair"], two["pair"]]
    cons = [lone["cons"], two["cons"]] if lone["cons"] else None
    energies = [lone["energies"], two["energies"]] if lone["energies"] else None
    stage = _stage_env(monkeypatch, {}, model0)
    try:
        smp, _, _, _ = _sampled(stage, pairs, opts(), 100000, 4, cons, energies, ("s1", "co"))
    finally:
        stage.close()
    check_distribution(smp[0]["s1"], exact_distribution(model0, sorc0, lone["seq"], 0, lone["allow"], lone["E"]))
    check_distribution(smp[1]["co"], exact_distribution(model0, sorc0, two["seq"], two["cp"], two["allow"], two["E"]))


@gpu
def test_gpu_marginals(sorc, bundled, monkeypatch):
    seqs = bundled["sequences"]
    s1, s2 = seqs["MicA"], seqs["ompA"]
    n1, n2 = len(s1), len(s2)
    N = 20000
    o = opts()
    stage = _stage_env(monkeypatch, {})
    try:
        smp, _, _, _ = _sampled(stage, [(s1, s2)], o, N, 99)
    finally:
        stage.close()

    def within(count, p):   # 6 sigma, plus 3 counts for the Poisson regime of pairs with N p << 1
        return np.abs(count - N * p) <= 6 * np.sqrt(N * p * (1 - p)) + 3

    for which, name, seq, cp in ((0, "s1", s1, 0), (1, "s2", s2, 0), (2, "co", s1 + s2, n1 + 1)):
        n = len(seq)
        pr, up, _ = sorc.fold(seq, cp, None, None, o.max_w if which < 2 else 0)
        t = smp[0][name].astype(np.int64)
        cnt = np.zeros((n + 1, n + 1))
        rows, cols = np.nonzero(t)
        i, j = cols + 1, t[rows, cols]
        keep = j > i
        np.add.at(cnt, (i[keep], j[keep]), 1)
        iu = np.triu_indices(n + 1, 1)
        assert np.all(within(cnt[iu], pr[iu])), name
        if which == 2:
            assert cnt[1:n1 + 1, n1 + 1:].sum() > 0   # inter-strand pairs were drawn and checked
            continue
        # unpaired windows: run[s, i] = unpaired bases from i on
        unp = (t == 0)
        run = np.zeros((N, n + 1), dtype=np.int64)
        for x in range(n - 1, -1, -1):
            run[:, x] = np.where(unp[:, x], run[:, x + 1] + 1, 0)
        for d in range(o.max_w):
            f = (run[:, :n] >= d + 1).sum(axis=0)
            ok = within(f[:n - d], up[:n - d, d])
            assert np.all(ok), (name, d)


@gpu
def test_gpu_byte_identity(sorc, bundled, monkeypatch):
    pairs, cons, energies = _bundled_data(bundled)
    o = opts()
    stage = _stage_env(monkeypatch, {})
    try:
        b = stage.batch(pairs, o, cons, energies)
        try:
            b.run()
            soft = b.fetch_dense().copy()
            soft_lz = b.fetch_logz()
        finally:
            b.close()
        _, _, lz0, flat0 = _sampled(stage, pairs, o, 0, 1, cons, energies)
        assert flat0.tobytes() == soft.tobytes() and lz0.tobytes() == soft_lz.tobytes()
        # co-fold samples of the pairs: the folds keep their bytes, the co-folds meet the oracle bar
        smp, res, lz, _ = _sampled(stage, pairs, o, 30, 5, cons, energies, ("co",))
        b = stage.batch(pairs, o, cons, energies)
        try:
            b.run()
            ref = b.split_dense(b.fetch_dense())
        finally:
            b.close()
        for k, (s1, s2) in enumerate(pairs):
            assert set(smp[k]) == {"co"}
            r, q = res[k], ref[k]
            for x in ("bp1", "up1", "bp2", "up2"):
                assert getattr(r, x).tobytes() == getattr(q, x).tobytes(), (k, x)
            assert lz[k][0] == soft_lz[k][0] and lz[k][1] == soft_lz[k][1]
            seq, cp, allow, E = _problem_inputs(s1, s2, 2, cons[k], energies[k])
            pr, _, olz = sorc.fold(seq, cp, allow, E, 0)
            n1, n2 = len(s1), len(s2)
            want = np.zeros((n1 + 1, n2 + 1))
            want[1:, 1:] = pr[1:n1 + 1, n1 + 1:]
            want = np.where((want >= o.th_hy) & (want.astype(np.float32) > np.float32(o.th_hy)), want, 0)
            np.testing.assert_allclose(r.hp, want, rtol=0, atol=TOL)
            assert abs(lz[k][2] - olz) < 1e-9
    finally:
        stage.close()


@gpu
def test_gpu_tensors_seeds_and_batches(bundled, monkeypatch):
    import torch
    seqs = bundled["sequences"]
    pairs = [(seqs[a], seqs[b]) for a, b in bundled["pairs"]]
    o = opts()
    stage = _stage_env(monkeypatch, {"RP_CLUSTER": "0"})
    try:
        b = stage.batch(pairs[:3], o, samples=12, sample_seed=8, sample_problems=("s1", "co"))
        try:
            b.run()
            host = b.fetch_samples()
            t = b.sample_tensors()
            torch.cuda.synchronize()
        finally:
            b.close()
        for k, (s1, s2) in enumerate(pairs[:3]):
            n1, n2 = len(s1), len(s2)
            assert np.array_equal(t["s1"][k, :, :n1].cpu().numpy(), host[k]["s1"])
            assert not t["s1"][k, :, n1:].any() and not t["s2"][k].any()
            assert np.array_equal(t["co"][k, :, :n1 + n2].cpu().numpy(), host[k]["co"])
            assert not t["co"][k, :, n1 + n2:].any()
        again, _, _, _ = _sampled(stage, pairs[:3], o, 12, 8, problems=("s1", "co"))
        other, _, _, _ = _sampled(stage, pairs[:3], o, 12, 9, problems=("s1", "co"))
        more, _, _, _ = _sampled(stage, pairs, o, 12, 8, problems=("s1", "co"))
        for k in range(3):
            for name in ("s1", "co"):
                assert np.array_equal(again[k][name], host[k][name])
                assert np.array_equal(more[k][name], host[k][name])
                assert not np.array_equal(other[k][name], host[k][name])
    finally:
        stage.close()


@gpu
def test_gpu_command_line(bundled, tmp_path):
    from ractip_b200 import ProbabilityStage, joint_structure
    seqs = bundled["sequences"]
    (tmp_path / "a.fa").write_text(f">MicA\n{seqs['MicA']}\n")
    (tmp_path / "b.fa").write_text(f">ompA\n{seqs['ompA']}\n")
    r = _cli(["--sample", "5", "--sample-seed", "3", str(tmp_path / "a.fa"), str(tmp_path / "b.fa")])
    assert r.returncode == 0, r.stdout
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 11
    stage = ProbabilityStage()
    try:
        b = stage.batch([(seqs["MicA"], seqs["ompA"])], opts(), samples=5, sample_seed=3, sample_problems=("co",))
        try:
            b.run()
            co = b.fetch_samples()[0]["co"]
        finally:
            b.close()
    finally:
        stage.close()
    assert lines[6:] == ["&".join(joint_structure(t, len(seqs["MicA"]))) for t in co]


# ------------------------------------------------------------------------------------------------ C++ shim
def _sample_check(tmp_path):
    exe = tmp_path / "sample_check"
    _cc(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", str(ROOT / "include"),
         str(ROOT / "tests" / "cpp" / "sample_check.cpp"), "-L", str(ROOT / "ractip_b200"), "-lractip_prob",
         f"-Wl,-rpath,{ROOT / 'ractip_b200'}", "-o", str(exe)])
    return exe


def test_cpp_shim_sampling_overload_compiles(lib, tmp_path):
    assert _sample_check(tmp_path).exists()


@gpu
@pytest.mark.parametrize("problem", [1, 2, 4], ids=["s1", "s2", "co"])
def test_gpu_cpp_shim_samples_equal_python(bundled, tmp_path, problem):
    from ractip_b200 import ProbabilityStage
    seqs = bundled["sequences"]
    s1, s2 = seqs["MicA"], seqs["ompA"]
    r = subprocess.run([str(_sample_check(tmp_path)), "gpu", s1, s2, str(problem), "7", "12"], stdout=subprocess.PIPE,
                       text=True)
    assert r.returncode == 0, r.stdout
    lines = r.stdout.strip().splitlines()
    got = np.array([[int(x) for x in l.split()] for l in lines[1:]], dtype=np.int16)
    name = {1: "s1", 2: "s2", 4: "co"}[problem]
    stage = ProbabilityStage()
    try:
        b = stage.batch([(s1, s2)], opts(), samples=7, sample_seed=12, sample_problems=(name,))
        try:
            b.run()
            want = b.fetch_samples()[0][name]
        finally:
            b.close()
    finally:
        stage.close()
    assert got.shape == want.shape and np.array_equal(got, want)


def test_sample_size_overflow_is_an_error(shim):
    """sizes past size_t are rejected by check_samples, not planned as a batch without samples"""
    huge = (RpPair * 4)()
    for k in range(4):
        huge[k].s1, huge[k].n1, huge[k].s2, huge[k].n2 = b"A", 2 ** 31 - 1, b"A", 2 ** 31 - 1
    msg = C.create_string_buffer(256)
    key = np.zeros(8, dtype=np.uint16)
    klen, same = C.c_longlong(), C.c_int()
    probs = np.zeros((12, 4), dtype=np.int64)
    o = opts()
    rc = shim.sample_shim(huge, None, None, 4, C.byref(o), C.byref(RpSampleOpts(2 ** 31 - 1, 1, 7)), msg, 256,
                          key.ctypes.data, C.byref(klen), 8, probs.ctypes.data, C.byref(same))
    assert rc == RP_ERR_ARG and "overflow the sample buffer's size" in msg.value.decode()


@pytest.mark.parametrize("cp", [0, 41], ids=["fold", "cofold"])
def test_oracle_sampler_marginals(sorc, cp):
    """Past the enumeration's reach (multiloops, nested multiloops, the nick's exterior loop): the oracle sampler's pair
    and unpaired-window frequencies on a 72-nt problem against the oracle's own probabilities, 6 sigma plus 3 counts
    for the Poisson regime of pairs with N p << 1"""
    rng = np.random.default_rng(61 + cp)
    n, N, w = 72, 20000, 8
    seq = rand_seq(rng, n, "GGCCAUAUGC")
    pr, up, _ = sorc.fold(seq, cp, None, None, 0 if cp else w)
    t = sorc.sample(seq, cp, None, None, seed=3, pair=0, kind=2 if cp else 0, num=N).astype(np.int64)

    def within(count, p):
        return np.abs(count - N * p) <= 6 * np.sqrt(N * p * (1 - p)) + 3

    cnt = np.zeros((n + 1, n + 1))
    rows, cols = np.nonzero(t)
    i, j = cols + 1, t[rows, cols]
    np.add.at(cnt, (i[j > i], j[j > i]), 1)
    iu = np.triu_indices(n + 1, 1)
    assert np.all(within(cnt[iu], pr[iu]))
    multi = 0   # samples with a multiloop: a pair enclosing two or more pairs side by side
    for row in t[:2000]:
        for a in range(1, n + 1):
            b = row[a - 1]
            if b > a:
                k, inner = a + 1, 0
                while k < b:
                    if row[k - 1] > k:
                        inner += 1
                        k = row[k - 1] + 1
                    else:
                        k += 1
                multi += inner >= 2
    assert multi > 100, multi   # the multiloop decisions were exercised
    if cp:
        assert cnt[1:cp, cp:].sum() > 0
        return
    unp = t == 0
    run = np.zeros((N, n + 1), dtype=np.int64)
    for x in range(n - 1, -1, -1):
        run[:, x] = np.where(unp[:, x], run[:, x + 1] + 1, 0)
    for d in range(w):
        assert np.all(within((run[:, :n] >= d + 1).sum(axis=0)[:n - d], up[:n - d, d])), d
