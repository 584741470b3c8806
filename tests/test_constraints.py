"""Structure constraints (-c): each problem of a pair keeps only the pairs its constraint allows.

The allowed-pair matrices here are written from the three rules of the contract (include/ractip_prob.h,
rp_constraint) by brute force; they share no code with the key derivation of ractip_b200/csrc/plan.cpp they check.
CPU: the masked oracle against exhaustive enumeration, the host derivation and routing, the general kernel's phase
functions in the host emulator, the front end's mapping.  GPU: the library against the masked oracle."""
import ctypes as C
import subprocess
import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

from ractip_b200._lib import RpConstraint, RpOpts, RpPair

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(Path(__file__).resolve().parent))
from conftest import rand_seq  # noqa: E402

TOL = 2e-7
RP_ERR_ARG = 1
TURN = 3
gpu = pytest.mark.gpu


# ----------------------------------------------------------------------------------------------- the contract
def _brackets(c, o, cl, base=0):
    st, out = [], []
    for i, ch in enumerate(c, 1):
        if ch == o:
            st.append(i)
        elif ch == cl:
            out.append((st.pop() + base, i + base))
    return out


def problem_view(c1, c2, n1, n2, which):
    """(length, bracket pairs, unpaired bases) of problem `which` (0: s1, 1: s2, 2: s1&s2), 1-based."""
    c1 = c1 if c1 is not None else "." * n1
    c2 = c2 if c2 is not None else "." * n2
    if which == 0:
        return n1, _brackets(c1, "(", ")"), {i for i, ch in enumerate(c1, 1) if ch in "x["}
    if which == 1:
        return n2, _brackets(c2, "(", ")"), {i for i, ch in enumerate(c2, 1) if ch in "x]"}
    opens = [i for i, ch in enumerate(c1, 1) if ch == "["][::-1]
    closes = [n1 + j for j, ch in enumerate(c2, 1) if ch == "]"]
    unp = {i for i, ch in enumerate(c1 + c2, 1) if ch in "x()"}
    return n1 + n2, list(zip(opens, closes)), unp


def allowed_matrix(m, pairs, unpaired):
    """allow[i, j] for 1 <= i < j <= m: neither base unpaired, a bracketed base only with its partner, no crossing."""
    partner = {}
    for p, q in pairs:
        partner[p], partner[q] = q, p
    A = np.zeros((m + 1, m + 1), dtype=np.uint8)
    for i in range(1, m + 1):
        for j in range(i + 1, m + 1):
            if i in unpaired or j in unpaired:
                continue
            if (i in partner or j in partner) and partner.get(i) != j:
                continue
            if any(p < i < q < j or i < p < j < q for p, q in pairs):
                continue
            A[i, j] = 1
    return A


def random_constraint(rng, n1, n2, dens=0.3):
    """A random valid (c1, c2): nested () within each string, nested [] across, some x."""
    def intra(n, reserve):
        c = ["."] * n
        free = [i for i in range(n) if i not in reserve]
        st = []
        for i in free:
            r = rng.random()
            if r < dens / 2 and len(st) < 6:
                st.append(i)
            elif r < dens and st and i - st[-1] > 1:
                c[st.pop()], c[i] = "(", ")"
            elif r < dens + 0.08:
                c[i] = "x"
        return c
    k = int(rng.integers(0, 4)) if n2 else 0
    left = sorted(rng.choice(n1, size=min(k, n1), replace=False)) if k else []
    right = sorted(rng.choice(n2, size=len(left), replace=False)) if k else []
    c1, c2 = intra(n1, set(left)), intra(n2, set(right))
    for i in left:
        c1[i] = "["
    for j in right:
        c2[j] = "]"
    return "".join(c1), "".join(c2)


# --------------------------------------------------------------------------------------------- masked oracle
class MaskedOracle:
    def __init__(self, so, model):
        self.lib = C.CDLL(str(so))
        vp, i = C.c_void_p, C.c_int
        self.lib.orc_params_new.restype = vp
        self.lib.orc_params_new.argtypes = [vp]
        self.lib.orc_set_maxloop.argtypes = [vp, i]
        for f in (self.lib.orc_fold_masked, self.lib.orc_enumerate_masked):
            f.restype = i
            f.argtypes = [vp, C.c_char_p, i, i, vp, vp, vp, i, vp]
        self._model = model
        self.P = self.lib.orc_params_new(C.addressof(model))

    def maxloop(self, m):
        self.lib.orc_set_maxloop(self.P, m)

    def _call(self, f, seq, cp, allow, max_w):
        n = len(seq)
        pr = np.zeros((n + 1, n + 1))
        up = np.zeros((n, max(max_w, 1)))
        lz = C.c_double()
        a = None if allow is None else np.ascontiguousarray(allow, dtype=np.uint8)
        rc = f(self.P, seq.encode(), n, cp, None if a is None else a.ctypes.data, pr.ctypes.data, up.ctypes.data,
               max_w, C.byref(lz))
        assert rc == 0
        return pr, (up if max_w > 0 else None), lz.value

    def fold(self, seq, cp=0, allow=None, max_w=0):
        return self._call(self.lib.orc_fold_masked, seq, cp, allow, max_w)

    def enumerate(self, seq, cp=0, allow=None, max_w=0):
        return self._call(self.lib.orc_enumerate_masked, seq, cp, allow, max_w)


def _cc(cmd):
    subprocess.run(cmd, check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)


@pytest.fixture(scope="module")
def morc(tmp_path_factory, model):
    so = tmp_path_factory.mktemp("morc") / "liboracle_masked.so"
    _cc(["gcc", "-O3", "-fPIC", "-shared", "-I", str(ROOT / "include"), str(ROOT / "tests" / "cpp" / "oracle_masked.c"),
         "-o", str(so), "-lm"])
    o = MaskedOracle(so, model)
    yield o
    o.maxloop(30)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = tmp_path_factory.mktemp("cshim") / "libconstraint_shim.so"
    csrc = ROOT / "ractip_b200" / "csrc"
    _cc(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", str(ROOT / "include"), "-I", str(csrc),
         str(csrc / "plan.cpp"), str(ROOT / "tests" / "cpp" / "constraint_shim.cpp"), "-o", str(so)])
    lib = C.CDLL(str(so))
    vp = C.c_void_p
    lib.constraint_shim.argtypes = [vp, vp, C.c_int, vp, C.c_char_p, C.c_int, vp, vp, C.c_int, vp]
    lib.constraint_shim.restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def kemul(tmp_path_factory):
    so = tmp_path_factory.mktemp("kemul") / "libemul_constrained.so"
    d = ROOT / "tests" / "emul"
    _cc(["g++", "-O2", "-U_FORTIFY_SOURCE", "-std=c++17", "-fPIC", "-shared", "-I", str(ROOT / "ractip_b200" / "csrc"),
         "-I", str(ROOT / "include"), "-o", str(so), str(d / "emul_constrained.cpp"),
         str(ROOT / "ractip_b200" / "csrc" / "dev_model.cpp")])
    lib = C.CDLL(str(so))
    vp, i = C.c_void_p, C.c_int
    lib.emul_constrained_problem.argtypes = [i, i, i, vp, vp, C.c_char_p, i, i, i, i, i, i, C.c_float, i, vp, vp, vp, vp]
    lib.emul_constrained_problem.restype = i
    return lib


def opts(**kw):
    o = dict(max_w=15, min_w=5, th_ss=0.5, th_hy=0.1, th_ac=0.003, use_pf_duplex=0)
    o.update(kw)
    return RpOpts(**o)


def plan_keys(shim, pairs, cons, o=None):
    """(rc, message, key buffer, per-problem (seq_off, n, constrained, general))"""
    keep = []
    arr = (RpPair * len(pairs))()
    carr = (RpConstraint * len(pairs))()
    for k, ((s1, s2), (c1, c2)) in enumerate(zip(pairs, cons)):
        b = [x.encode() if x is not None else None for x in (s1, s2, c1, c2)]
        keep.append(b)
        arr[k].s1, arr[k].n1, arr[k].s2, arr[k].n2 = b[0], len(s1), b[1] or None, len(s2)
        carr[k].c1, carr[k].c2 = b[2], b[3]
    cap = sum(2 * (len(a) + len(b)) + 4 for a, b in pairs) + 16
    key = np.zeros(cap, dtype=np.uint16)
    klen = C.c_longlong()
    probs = np.zeros((3 * len(pairs), 4), dtype=np.int64)
    msg = C.create_string_buffer(256)
    o = o or opts()
    rc = shim.constraint_shim(arr, carr, len(pairs), C.byref(o), msg, 256, key.ctypes.data, C.byref(klen), cap,
                              probs.ctypes.data)
    return rc, msg.value.decode(), key[:klen.value], probs


def key_matrix(keys, off, m):
    k = keys[off - 1:off + m].astype(np.int64)   # k[1..m] = the problem's keys
    A = np.zeros((m + 1, m + 1), dtype=np.uint8)
    for i in range(1, m + 1):
        A[i, i + 1:] = k[i + 1:] == k[i]
    return A


# --------------------------------------------------------------------------- masked oracle vs enumeration (CPU)
def _check_enum(morc, seq, cp, allow, max_w):
    pr, up, lz = morc.fold(seq, cp, allow, max_w)
    epr, eup, elz = morc.enumerate(seq, cp, allow, max_w)
    assert abs(lz - elz) < 1e-12 * max(1.0, abs(elz))
    np.testing.assert_allclose(pr, epr, rtol=0, atol=1e-12)
    if max_w:
        np.testing.assert_allclose(up, eup, rtol=0, atol=1e-12)
    if allow is not None:
        iu = np.triu_indices(len(seq) + 1, 1)
        assert np.all(pr[iu][allow[iu] == 0] == 0)


SINGLE = [("GGGAAACCCAGGGAAACCC", "x.................."),          # one base kept unpaired
          ("GGGAAACCCAGGGAAACCC", "(.......).........."),          # a bracket pair
          ("GGGGAAAUCCCCAGCUAGC", "..((....)).....x..."),
          ("AAAAGGGAAAACCCAAAAA", "(.................)"),         # A.A: a bracket pair that cannot form
          ("GCGCAAAAGCGCAAAAGCG", "((...)).((....))...")]


@pytest.mark.parametrize("maxloop", [30, 3])
def test_masked_oracle_single_strand(morc, maxloop):
    morc.maxloop(maxloop)
    try:
        rng = np.random.default_rng(11)
        cases = list(SINGLE)
        for _ in range(6):
            n = int(rng.integers(12, 19))
            cases.append((rand_seq(rng, n), random_constraint(rng, n, 0)[0]))
        for s, c in cases:
            m, pairs, unp = problem_view(c, None, len(s), 0, 0)
            _check_enum(morc, s, 0, allowed_matrix(m, pairs, unp), 6)
    finally:
        morc.maxloop(30)


@pytest.mark.parametrize("maxloop", [30, 3])
def test_masked_oracle_two_strands(morc, maxloop):
    morc.maxloop(maxloop)
    try:
        rng = np.random.default_rng(12)
        cases = [("GGGAAUCC", "GGAUUCCC", "..[[....", "....]]..", 2),      # [] alone
                 ("GGGAAUCC", "GGAUUCCC", "x.......", "....x...", 2),      # x alone
                 ("GCAAAAGCGG", "CCGAAAA", "(....)..[.", "..]....", 2),    # [] next to a () helix
                 ("GGCGAAAGCC", "GGCUUU", "((.[..).).", "...]..", 2)]      # [] inside a () helix
        for _ in range(6):
            n1, n2 = int(rng.integers(6, 10)), int(rng.integers(6, 9))
            s1, s2 = rand_seq(rng, n1), rand_seq(rng, n2)
            c1, c2 = random_constraint(rng, n1, n2)
            cases.append((s1, s2, c1, c2, 0))
        for s1, s2, c1, c2, _ in cases:
            n1, n2 = len(s1), len(s2)
            for which in (0, 1, 2):
                m, pairs, unp = problem_view(c1, c2, n1, n2, which)
                seq = (s1, s2, s1 + s2)[which]
                _check_enum(morc, seq, n1 + 1 if which == 2 else 0, allowed_matrix(m, pairs, unp), 0 if which == 2 else 5)
    finally:
        morc.maxloop(30)


def test_masked_oracle_inside_helix_is_nested(morc):
    """A kissing '[' inside a () helix: each problem sees one kind of bracket, so neither crosses the other."""
    c1 = "((((.(((((((..[[[[[[.)))))))...))))"
    m, pairs, unp = problem_view(c1, "((((.(((((((..]]]]]].)))))))...))))", 35, 35, 2)
    assert len(pairs) == 6 and all(c1[p - 1] == "[" for p, _ in pairs)
    A = allowed_matrix(m, pairs, unp)
    assert A[15, 35 + 20] == 1 and A[20, 35 + 15] == 1 and A[15, 35 + 15] == 0


# -------------------------------------------------------------------------------- host derivation (CPU)
def test_keys_equal_brute_force(shim):
    rng = np.random.default_rng(21)
    pairs, cons = [], []
    for _ in range(12):
        n1, n2 = int(rng.integers(5, 60)), int(rng.integers(0, 50))
        pairs.append((rand_seq(rng, n1), rand_seq(rng, n2)))
        cons.append(random_constraint(rng, n1, n2, dens=float(rng.choice([0.1, 0.3, 0.6]))))
        if n2 == 0:
            cons[-1] = (cons[-1][0], None)
    rc, msg, keys, probs = plan_keys(shim, pairs, cons)
    assert rc == 0, msg
    for p, ((s1, s2), (c1, c2)) in enumerate(zip(pairs, cons)):
        for which in (0, 1, 2):
            seq_off, n, constrained, general = probs[3 * p + which]
            if which == 2 and not s2:
                continue
            m, bp, unp = problem_view(c1, c2, len(s1), len(s2), which)
            want = allowed_matrix(m, bp, unp)
            full = np.triu(np.ones((m + 1, m + 1), dtype=np.uint8), 1)
            full[0, :] = 0
            restricts = bool(np.any(want != full))
            assert constrained == restricts, (p, which)
            if constrained:
                np.testing.assert_array_equal(key_matrix(keys, seq_off, m), want, err_msg=f"pair {p} problem {which}")
                assert general


BAD = [
    (("GGGAAACCC", "GGG"), ("....", None), "c1, position 5"),             # shorter
    (("GGGAAACCC", "GGG"), ("..........", None), "c1, position 10"),      # longer
    (("GGGAAACCC", "GGG"), ("...l.....", None), "c1, position 4"),        # outside .x()[]
    (("GGGAAACCC", "GGG"), ("((.....).", None), "c1, position 1"),        # '(' never closed
    (("GGGAAACCC", "GGG"), (")........", None), "c1, position 1"),        # ')' closes nothing
    (("GGGAAACCC", "GGG"), ("..[..[...", "..]"), "c1, position 3"),       # two '[', one ']'
    (("GGGAAACCC", "GGG"), (".........", "]]."), "c2, position 1"),       # ']' without '['
    (("GGGAAACCC", ""), ("..[......", None), "c1, position 3"),           # '[' with no second strand
    (("GGGAAACCC", "GGG"), ("..]......", None), "c1, position 3"),        # ']' in c1
    (("GGGAAACCC", "GGG"), (".........", ".[."), "c2, position 2"),       # '[' in c2
]


@pytest.mark.parametrize("pair,con,where", BAD)
def test_malformed_constraints(shim, pair, con, where):
    rc, msg, _, _ = plan_keys(shim, [("ACGU" * 5, "ACGU"), pair], [(None, None), con])
    assert rc == RP_ERR_ARG
    assert msg.startswith("pair 1, " + where), msg


def test_routing(shim):
    """Constrained problems go to the general kernel, the others are planned as without constraints."""
    pairs = [("ACGU" * 18, "ACGU" * 34)] * 3
    cons = [(None, None), ("(" + "." * 70 + ")", None), ("." * 72, "." * 136)]
    rc, msg, keys, probs = plan_keys(shim, pairs, cons)
    assert rc == 0, msg
    flags = probs[:, 2].tolist()
    assert flags == [0, 0, 0, 1, 0, 1, 0, 0, 0]   # pair 1: s1 and the co-fold ('(' ')' unpaired there)
    assert probs[:, 3].tolist() == flags           # these lengths run on the band kernel when unconstrained
    rc, _, keys0, probs0 = plan_keys(shim, pairs, [(None, None)] * 3)
    assert rc == 0 and len(keys0) == 0 and not probs0[:, 2].any() and not probs0[:, 3].any()
    rc, _, _, probs_d = plan_keys(shim, pairs, cons, opts(use_pf_duplex=1))
    assert probs_d[5, 2] == 0                      # --duplex: the hybridization stays unconstrained


# ------------------------------------------------------------------------------------------ emulator (CPU)
ROUTES = [(0, 1), (5, 1), (10, 1), (15, 1), (10, 8), (10, 16)]


def _emul(kemul, model, keys, seq, cp, kind, max_w, n1, n2, route, G, lockstep, T=64):
    n = len(seq)
    bp = np.zeros((n + 1) * (n + 2) // 2, dtype=np.float32)
    up = np.zeros((n, max(max_w, 1)), dtype=np.float32)
    hp = np.zeros((n1 + 1, n2 + 1), dtype=np.float32)
    lz = C.c_double()
    k = np.ascontiguousarray(keys, dtype=np.uint16)
    rc = kemul.emul_constrained_problem(route, G, int(lockstep), k.ctypes.data, C.addressof(model), seq.encode(), n, cp,
                                        kind, max_w, n1, n2, 0.1, T, bp.ctypes.data, up.ctypes.data, hp.ctypes.data,
                                        C.byref(lz))
    assert rc == 0, rc
    return bp, up, hp, lz.value


def _bp_matrix(bp, n):
    P = np.zeros((n + 1, n + 1))
    for i in range(1, n + 1):
        off = i * (2 * n + 1 - i) // 2
        P[i, i + 1:] = bp[off + i + 1:off + n + 1]
    return P


@pytest.mark.parametrize("lockstep", [False, True])
def test_emulator_routes(shim, kemul, morc, model, lockstep):
    rng = np.random.default_rng(31)
    s1, s2 = rand_seq(rng, 47), rand_seq(rng, 38)
    c1, c2 = random_constraint(rng, 47, 38)
    rc, msg, keys, probs = plan_keys(shim, [(s1, s2)], [(c1, c2)])
    assert rc == 0, msg
    for route, G in ROUTES:
        for which in (0, 2):
            seq_off, n, con, _ = probs[which]
            m, bp, unp = problem_view(c1, c2, 47, 38, which)
            allow = allowed_matrix(m, bp, unp)
            k = keys[seq_off - 1:seq_off + m]
            if which == 0:
                b, u, _, lz = _emul(kemul, model, k, s1, 0, 0, 8, 47, 0, route, G, lockstep)
                pr, oup, olz = morc.fold(s1, 0, allow, 8)
                np.testing.assert_allclose(_bp_matrix(b, 47), pr, rtol=0, atol=TOL)
                np.testing.assert_allclose(u, oup, rtol=0, atol=TOL)
            else:
                _, _, h, lz = _emul(kemul, model, k, s1 + s2, 48, 1, 0, 47, 38, route, G, lockstep)
                pr, _, olz = morc.fold(s1 + s2, 48, allow, 0)
                want = pr[:48, 47:]   # rows i <= n1, columns j = n1 + 1 .. n1 + n2 (hp[i][j - n1])
                o = np.zeros((48, 39))
                o[1:, 1:] = want[1:, 1:]
                o = np.where((o >= 0.1) & (o.astype(np.float32) > np.float32(0.1)), o, 0)
                np.testing.assert_allclose(h, o, rtol=0, atol=TOL)
            assert abs(lz - olz) < 1e-10, (route, G, which)


# ------------------------------------------------------------------------------------------ front end (CPU)
def test_constraint_line():
    from ractip_b200.frontend import FastaRecord, constraint_line
    assert constraint_line(FastaRecord("a", "ACGU", "")) is None
    assert constraint_line(FastaRecord("a", "ACGUA", "(? ).")) == "(..)."
    with pytest.raises(ValueError, match="'l' at position 2"):
        constraint_line(FastaRecord("a", "ACGU", ".l.."))
    with pytest.raises(ValueError, match="'e'"):
        constraint_line(FastaRecord("a", "ACGU", "...e"))
    with pytest.raises(ValueError, match="3 characters"):
        constraint_line(FastaRecord("a", "ACGU", "..."))


def test_predict_leaves_shuffles_unconstrained(monkeypatch):
    """-c constrains the original pairs' batch; the z-score shuffles have no structure line."""
    from ractip_b200 import frontend
    from ractip_b200.frontend import FastaRecord
    calls = []

    class Stop(Exception):
        pass

    class FakeStage:
        model = None

        def run_dense(self, seqs, opts, constraints=None):
            calls.append((list(seqs), constraints))
            if len(calls) == 2:
                raise Stop
            return [SimpleNamespace(bp1=None, bp2=None) for _ in seqs]

    monkeypatch.setattr(frontend, "solve_joint", lambda *a, **k: None)
    monkeypatch.setattr(frontend, "solve_ss", lambda *a, **k: (None, None, 0.0))
    a, b = FastaRecord("a", "GGGAAACCC", "x?.(...)."), FastaRecord("b", "GGGUUUCCC", "")
    with pytest.raises(Stop):
        frontend.predict(FakeStage(), [(a, b)], zscore=12, num_shuffling=3, use_constraint=True)
    assert calls[0][1] == [("x..(...).", None)]
    assert len(calls[1][0]) == 3 and calls[1][1] is None
    calls.clear()
    with pytest.raises(Stop):
        frontend.predict(FakeStage(), [(a, b)], zscore=12, num_shuffling=3)
    assert calls[0][1] is None   # without -c the structure lines are ignored


# ------------------------------------------------------------------------------------------------- GPU
def _stage_env(monkeypatch, env):
    from ractip_b200 import ProbabilityStage
    for k in ("RP_BAND", "RP_CLUSTER", "RP_MCC_LONG_N"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    return ProbabilityStage()


def _oracle_pair(morc, s1, s2, c1, c2, o):
    n1, n2 = len(s1), len(s2)
    out = {}
    for which, seq in ((0, s1), (1, s2)):
        m, bp, unp = problem_view(c1, c2, n1, n2, which)
        A = allowed_matrix(m, bp, unp)
        out[which] = morc.fold(seq, 0, A, o.max_w) + (A,)
    m, bp, unp = problem_view(c1, c2, n1, n2, 2)
    A = allowed_matrix(m, bp, unp)
    out[2] = morc.fold(s1 + s2, n1 + 1, A, 0) + (A,)
    return out


def _compare(r, lz, orc, n1, n2, o):
    for which, (bp, nn) in ((0, (r.bp1, n1)), (1, (r.bp2, n2))):
        pr, up, olz, A = orc[which]
        got = _bp_matrix(bp, nn)
        np.testing.assert_allclose(got, pr, rtol=0, atol=TOL)
        iu = np.triu_indices(nn + 1, 1)
        assert np.all(got[iu][A[iu] == 0] == 0)
        np.testing.assert_allclose((r.up1, r.up2)[which], up, rtol=0, atol=TOL)
        assert abs(lz[which] - olz) < 1e-9
    pr, _, olz, A = orc[2]
    want = np.zeros((n1 + 1, n2 + 1))
    want[1:, 1:] = pr[1:n1 + 1, n1 + 1:]
    want = np.where((want >= o.th_hy) & (want.astype(np.float32) > np.float32(o.th_hy)), want, 0)
    np.testing.assert_allclose(r.hp, want, rtol=0, atol=TOL)
    assert np.all(r.hp[1:, 1:][A[1:n1 + 1, n1 + 1:] == 0] == 0)
    assert abs(lz[2] - olz) < 1e-9


def _run(stage, pairs, cons, o):
    b = stage.batch(pairs, o, cons)
    try:
        b.run()
        flat = b.fetch_dense()
        return b.split_dense(flat), b.fetch_logz(), flat.copy()
    finally:
        b.close()


@gpu
def test_gpu_bundled_pairs(morc, bundled, monkeypatch):
    seqs, dis = bundled["sequences"], bundled["readme_dis"]
    rng = np.random.default_rng(41)
    pairs, cons = [(seqs["DIS"], seqs["DIS"])], [(dis["s1"], dis["s2"])]
    for a, b in (("MicA", "ompA"), ("OxyS", "fhlA"), ("CopA", "CopT")):
        pairs.append((seqs[a], seqs[b]))
        cons.append(random_constraint(rng, len(seqs[a]), len(seqs[b]), dens=0.15))
    o = opts()
    stage = _stage_env(monkeypatch, {})
    try:
        res, lz, _ = _run(stage, pairs, cons, o)
        for (s1, s2), (c1, c2), r, z in zip(pairs, cons, res, lz):
            _compare(r, z, _oracle_pair(morc, s1, s2, c1, c2, o), len(s1), len(s2), o)
        # sparse lists and tensors of the constrained batch agree with its dense fetch
        recs = stage.run_sparse(pairs, o, constraints=cons)
        for (s1, s2), r, sp in zip(pairs, res, recs):
            n1, n2 = len(s1), len(s2)
            P1 = _bp_matrix(r.bp1, n1)
            want_x = sorted((i - 1, j - 1) for i in range(1, n1 + 1) for j in range(i + 1, n1 + 1) if P1[i, j] > o.th_ss)
            assert sorted((int(x["i"]), int(x["j"])) for x in sp.x) == want_x
            want_z = sorted((i - 1, j - 1) for i in range(1, n1 + 1) for j in range(1, n2 + 1) if r.hp[i, j] > o.th_hy)
            assert sorted((int(x["i"]), int(x["j"])) for x in sp.z) == want_z
        import torch
        b = stage.batch(pairs, o, cons)
        try:
            b.run()
            t = b.tensors()
            torch.cuda.synchronize()
            for k, r in enumerate(res):
                n1, n2 = len(pairs[k][0]), len(pairs[k][1])
                np.testing.assert_array_equal(t["hp"][k, :n1 + 1, :n2 + 1].cpu().numpy(), r.hp)
                np.testing.assert_array_equal(np.triu(t["bp1"][k, :n1 + 1, :n1 + 1].cpu().numpy(), 1),
                                              _bp_matrix(r.bp1, n1).astype(np.float32))
        finally:
            b.close()
    finally:
        stage.close()


ROUTE_ENVS = [{}, {"RP_MCC_LONG_N": "1", "RP_CLUSTER": "0"}, {"RP_CLUSTER": "8"}, {"RP_CLUSTER": "16"}]


@gpu
@pytest.mark.parametrize("env", ROUTE_ENVS, ids=["default", "wide", "cluster8", "cluster16"])
def test_gpu_long_pair_routes(morc, monkeypatch, env):
    rng = np.random.default_rng(42)
    s1, s2 = rand_seq(rng, 620), rand_seq(rng, 300)
    c1, c2 = random_constraint(rng, 620, 300, dens=0.05)
    o = opts()
    stage = _stage_env(monkeypatch, env)
    try:
        res, lz, _ = _run(stage, [(s1, s2)], [(c1, c2)], o)
    finally:
        stage.close()
    _compare(res[0], lz[0], _oracle_pair(morc, s1, s2, c1, c2, o), 620, 300, o)


@gpu
def test_gpu_all_dots_and_mixed_batch(bundled, monkeypatch):
    seqs = bundled["sequences"]
    pairs = [(seqs[a], seqs[b]) for a, b in (("MicA", "ompA"), ("DIS", "DIS"), ("OxyS", "fhlA"))]
    o = opts()
    stage = _stage_env(monkeypatch, {"RP_BAND": "0"})
    try:
        dots = [("." * len(a), "." * len(b)) for a, b in pairs]
        _, lz0, plain = _run(stage, pairs, None, o)
        _, lz1, con = _run(stage, pairs, dots, o)
        assert plain.tobytes() == con.tobytes() and lz0.tobytes() == lz1.tobytes()
    finally:
        stage.close()
    stage = _stage_env(monkeypatch, {})
    try:
        dis = bundled["readme_dis"]
        mixed = [None, (dis["s1"], dis["s2"]), None]
        r0, lz0, _ = _run(stage, pairs, None, o)
        r1, lz1, _ = _run(stage, pairs, mixed, o)
        for k in (0, 2):
            for f in ("bp1", "bp2", "up1", "up2", "hp"):
                assert getattr(r0[k], f).tobytes() == getattr(r1[k], f).tobytes()
            assert lz0[k].tobytes() == lz1[k].tobytes()
        # --duplex: the hybridization ignores the constraint
        od = opts(use_pf_duplex=1)
        d0, _, _ = _run(stage, pairs, None, od)
        d1, _, _ = _run(stage, pairs, mixed, od)
        assert d0[1].hp.tobytes() == d1[1].hp.tobytes()
    finally:
        stage.close()


@gpu
def test_gpu_command_line(bundled, tmp_path):
    seqs, dis = bundled["sequences"], bundled["readme_dis"]
    c1 = "xxxx" + dis["s1"][4:-4] + "xxxx"   # the outer helix's four pairs: both ends kept unpaired
    (tmp_path / "a.fa").write_text(f">a\n{seqs['DIS']}\n{c1}\n")
    (tmp_path / "b.fa").write_text(f">b\n{seqs['DIS']}\n{dis['s2']}\n")
    r = subprocess.run([sys.executable, "-m", "ractip_b200", "-c", str(tmp_path / "a.fa"), str(tmp_path / "b.fa")],
                       cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout
    lines = r.stdout.splitlines()
    assert lines[0] == ">a" and len(lines[2]) == 35
    assert lines[2][:4] == "...." and lines[2][-4:] == "...."   # the x bases get no pair
    (tmp_path / "c.fa").write_text(f">c\n{seqs['DIS']}\n{'.l' + c1[2:]}\n")
    r = subprocess.run([sys.executable, "-m", "ractip_b200", "-c", str(tmp_path / "c.fa"), str(tmp_path / "b.fa")],
                       cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 1 and "'l' at position 2" in r.stdout
