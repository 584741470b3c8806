"""Parity of the CUDA probability stage (through the C ABI) with the CPU oracle.

Bars (BASELINE.json north_star): every probability within 1e-6 absolute of the fp64
reference path; identical thresholded variable sets.  The outputs are fp32 casts of fp64
values (src/ractip.cpp:367,375,453), so agreement is checked at float resolution:
|diff| <= 2e-7 on values in [0,1] (one fp32 ulp at 1.0 is 1.2e-7), far inside the 1e-6 bar.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import rand_seq

pytestmark = pytest.mark.gpu

TOL = 2e-7          # fp32 ulp-level; the north_star bar is 1e-6
BAR = 1e-6


def _oracle_pair(oracle, s1, s2, opts):
    bp1, up1 = oracle.rnafold(s1, opts.max_w)
    bp2, up2 = oracle.rnafold(s2, opts.max_w)
    hp = oracle.rnaduplex(s1, s2, opts.th_hy, bool(opts.use_pf_duplex))
    return bp1, up1, bp2, up2, hp


def _threshold_sets(bp1, up1, bp2, up2, hp, n1, n2, opts):
    """Variable lists in the reference's creation order (src/ractip.cpp:557-567,578-588,598-609,621-627)."""
    def xs(bp, L):
        out = []
        off = [i * (2 * L + 1 - i) // 2 for i in range(L + 1)]
        for j in range(1, L):
            for i in range(j - 1, -1, -1):
                if bp[off[i + 1] + j + 1] > np.float32(opts.th_ss):
                    out.append((i, j))
        return out
    z = [(i, j) for i in range(n1) for j in range(n2) if hp[i + 1][j + 1] > np.float32(opts.th_hy)]
    def vs(up):
        return [(i, i + j) for i in range(up.shape[0]) for j in range(opts.min_w - 1, up.shape[1])
                if up[i][j] > np.float32(opts.th_ac)]
    return xs(bp1, n1), xs(bp2, n2), z, vs(up1), vs(up2)


def _near_threshold(a, th, eps=3e-7):
    return np.abs(a.astype(np.float64) - float(np.float32(th))) < eps


def _compare(res, ora, s1, s2, opts, tag=""):
    bp1, up1, bp2, up2, hp = ora
    for name, got, want in [("bp1", res.bp1, bp1), ("bp2", res.bp2, bp2), ("up1", res.up1, up1), ("up2", res.up2, up2)]:
        d = np.abs(got.astype(np.float64) - want.astype(np.float64)).max() if got.size else 0.0
        assert d <= TOL, (tag, name, d)
    # hp is thresholded: entries within float noise of th_hy may legitimately differ in presence
    mism = (res.hp != 0) != (hp != 0)
    if mism.any():
        dense = np.where(res.hp != 0, res.hp, hp)
        assert _near_threshold(dense[mism], opts.th_hy).all(), (tag, "hp support")
    both = (res.hp != 0) & (hp != 0)
    if both.any():
        assert np.abs(res.hp[both].astype(np.float64) - hp[both]).max() <= TOL, (tag, "hp")


def test_bundled_pairs_one_ragged_batch(stage, oracle, bundled):
    """All 8 bundled pairs (SURVEY.md 4) in one call: dense parity and identical variable sets."""
    from ractip_b200 import default_opts
    opts = default_opts()
    pairs = [(bundled["sequences"][a], bundled["sequences"][b]) for a, b in bundled["pairs"]]
    res = stage.run_dense(pairs, opts)
    assert stage.last_timing().kernel_launches >= 1
    for (a, b), (s1, s2), r in zip(bundled["pairs"], pairs, res):
        ora = _oracle_pair(oracle, s1, s2, opts)
        _compare(r, ora, s1, s2, opts, f"{a}x{b}")
        got = _threshold_sets(r.bp1, r.up1, r.bp2, r.up2, r.hp, len(s1), len(s2), opts)
        want = _threshold_sets(*ora, len(s1), len(s2), opts)
        for g, w, nm, arr, th in zip(got, want, "xyzvw", (r.bp1, r.bp2, r.hp, r.up1, r.up2),
                                     (opts.th_ss, opts.th_ss, opts.th_hy, opts.th_ac, opts.th_ac)):
            if g != w:  # only values sitting on the threshold within float noise may flip
                assert _near_threshold(np.asarray(arr).ravel(), th).any(), (a, b, nm)
            else:
                assert g == w
        assert np.array_equal(r.offset1, np.array([i * (2 * len(s1) + 1 - i) // 2 for i in range(len(s1) + 1)]))


def test_readme_dis_known_answer_on_gpu(stage, bundled):
    """README.md:91-97: the thresholded GPU matrices contain exactly the answer's helices."""
    s = bundled["sequences"]["DIS"]
    r = stage.solve_probabilities(s, s)
    ans = bundled["readme_dis"]["s1"]
    stack, want = [], set()
    for k, ch in enumerate(ans):
        if ch == "(":
            stack.append(k)
        elif ch == ")":
            want.add((stack.pop(), k))
    L = len(s)
    got = {(i, j) for j in range(1, L) for i in range(j) if r.bp1[r.offset1[i + 1] + j + 1] > 0.5}
    assert got == want
    kiss = [k for k, ch in enumerate(ans) if ch == "["]
    for a, b in zip(kiss, reversed(kiss)):
        assert r.hp[a + 1][b + 1] > 0.9


@pytest.mark.parametrize("n1,n2", [(1, 1), (2, 5), (4, 4), (5, 5), (7, 3), (9, 12), (33, 64), (130, 31)])
def test_edge_and_ragged_lengths(stage, oracle, n1, n2):
    from ractip_b200 import default_opts
    rng = np.random.default_rng(1000 * n1 + n2)
    opts = default_opts()
    pairs = [(rand_seq(rng, n1), rand_seq(rng, n2)) for _ in range(3)]
    for (s1, s2), r in zip(pairs, stage.run_dense(pairs, opts)):
        _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, f"{n1}x{n2}")


def test_longer_than_one_cta_chunk(stage, oracle):
    """n > CTA width: the per-diagonal cell loop runs in several chunks (two-strand n = 430)."""
    from ractip_b200 import default_opts
    rng = np.random.default_rng(77)
    s1, s2 = rand_seq(rng, 300), rand_seq(rng, 130)
    opts = default_opts()
    r = stage.run_dense([(s1, s2)], opts)[0]
    _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, "300x130")


def test_options_window_thresholds(stage, oracle, bundled):
    from ractip_b200 import default_opts
    s1, s2 = bundled["sequences"]["Tar"], bundled["sequences"]["Tarstar"]
    for kw in [dict(max_w=1), dict(max_w=30, min_w=3), dict(th_hy=0.0), dict(th_hy=0.5, th_ss=0.2)]:
        opts = default_opts(**kw)
        r = stage.run_dense([(s1, s2)], opts)[0]
        assert r.up1.shape == (len(s1), opts.max_w)
        _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, str(kw))


def test_special_hairpins_and_letters(stage, oracle):
    from ractip_b200 import default_opts
    opts = default_opts()
    pairs = [("GGGGGACCCC", "CCAACGGG"), ("ggggaccuuaugc", "GGGTGACTCC"), ("ACAGUACUGAGCAGUACU", "NNACGUNNACGU")]
    for (s1, s2), r in zip(pairs, stage.run_dense(pairs, opts)):
        _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, s1)


def test_pf_duplex_branch(stage, oracle, bundled):
    """--duplex (src/ractip.cpp:390-399): dense hp from the log-space duplex forward/backward."""
    from ractip_b200 import default_opts
    opts = default_opts(use_pf_duplex=1)
    pairs = [(bundled["sequences"]["DIS"], bundled["sequences"]["DIS"]),
             (bundled["sequences"]["MicA"], bundled["sequences"]["ompA"]), ("GGGAAACC", "GGUUUCCC"), ("A", "U")]
    for (s1, s2), r in zip(pairs, stage.run_dense(pairs, opts)):
        want = oracle.rnaduplex(s1, s2, opts.th_hy, True)
        assert np.abs(r.hp.astype(np.float64) - want).max() <= TOL
        bp1, up1 = oracle.rnafold(s1, opts.max_w)
        assert np.abs(r.bp1 - bp1).max() <= TOL and np.abs(r.up1 - up1).max() <= TOL


def test_log_partition_functions(stage, oracle, bundled):
    from ractip_b200 import default_opts
    s1, s2 = bundled["sequences"]["CopA"], bundled["sequences"]["CopT"]
    b = stage.batch([(s1, s2)], default_opts())
    b.run()
    lz = b.fetch_logz()[0]
    b.close()
    want = [oracle.fold(s1)[2], oracle.fold(s2)[2], oracle.fold(s1 + s2, len(s1) + 1)[2]]
    assert np.abs(lz - np.array(want)).max() < 1e-9


def test_sparse_records_in_reference_order(stage, oracle, bundled):
    """rp_run_sparse == thresholding the dense matrices in the reference's loop order."""
    from ractip_b200 import default_opts
    opts = default_opts()
    pairs = [(bundled["sequences"][a], bundled["sequences"][b]) for a, b in bundled["pairs"]]
    dense = stage.run_dense(pairs, opts)
    sparse = stage.run_sparse(pairs, opts)
    for (s1, s2), d, sp in zip(pairs, dense, sparse):
        x, y, z, _, _ = _threshold_sets(d.bp1, d.up1, d.bp2, d.up2, d.hp, len(s1), len(s2), opts)
        assert [(int(r["i"]), int(r["j"])) for r in sp.x] == x
        assert [(int(r["i"]), int(r["j"])) for r in sp.y] == y
        assert [(int(r["i"]), int(r["j"])) for r in sp.z] == z
        for r in sp.x:
            assert r["p"] == d.bp1[d.offset1[r["i"] + 1] + r["j"] + 1]
        for r in sp.z:
            assert r["p"] == d.hp[r["i"] + 1][r["j"] + 1]
        assert np.array_equal(sp.up1, d.up1) and np.array_equal(sp.up2, d.up2)


def test_shuffle_batch_matches_oracle_and_is_deterministic(stage, oracle, bundled):
    """A slice of the --zscore batch (MicA x ompA, seed 1) against the oracle; bitwise repeatable."""
    from ractip_b200 import default_opts, zscore_shuffles
    s1, s2 = bundled["sequences"]["MicA"], bundled["sequences"]["ompA"]
    r1, r2 = zscore_shuffles(s1, s2, 12, 1)
    pairs = list(zip(r1, r2))
    opts = default_opts()
    b = stage.batch(pairs, opts)
    b.run()
    flat1 = b.fetch_dense().copy()
    b.run()
    flat2 = b.fetch_dense().copy()
    assert np.array_equal(flat1, flat2)
    for (a, c), r in zip(pairs, b.split_dense(flat1)):
        _compare(r, _oracle_pair(oracle, a, c, opts), a, c, opts, "shuffle")
    b.close()


def test_full_batch_size_independent_properties(stage, bundled):
    """BASELINE config 4 at full size (1000 shuffles): properties that need no oracle.
    sum_j p(i,j) + P(i unpaired) = 1 for every base of every shuffled sequence; windows monotone;
    hp entries either 0 or above the threshold; dinucleotide-shuffled inputs keep their length."""
    from ractip_b200 import default_opts, zscore_shuffles
    s1, s2 = bundled["sequences"]["MicA"], bundled["sequences"]["ompA"]
    r1, r2 = zscore_shuffles(s1, s2, 1000, 1)
    opts = default_opts()
    b = stage.batch(list(zip(r1, r2)), opts)
    b.run()
    flat = b.fetch_dense().copy()
    b.run()
    assert np.array_equal(flat, b.fetch_dense()), "the 3000-problem batch is not bitwise repeatable (a race?)"
    res = b.split_dense(flat)
    b.close()
    assert np.isfinite(flat).all()
    worst = 0.0
    for r in res:
        for bp, off, up in ((r.bp1, r.offset1, r.up1), (r.bp2, r.offset2, r.up2)):
            L = up.shape[0]
            full = np.zeros((L + 1, L + 1), dtype=np.float64)
            for i in range(1, L):
                full[i, i + 1:L + 1] = bp[off[i] + i + 1: off[i] + L + 1]
            tot = (full + full.T)[1:, 1:].sum(axis=1) + up[:, 0]
            worst = max(worst, np.abs(tot - 1).max())
            assert (np.diff(up.astype(np.float64), axis=1) <= 1e-6).all()
        nz = r.hp[r.hp != 0]
        assert (nz > np.float32(opts.th_hy)).all()
    assert worst < 5e-6  # ~L fp32 roundings per row


def test_error_paths(stage, lib):
    from ractip_b200 import default_opts, RpError
    from ractip_b200._lib import RpPair
    opts = default_opts()
    pairs = (RpPair * 1)()
    pairs[0].s1, pairs[0].n1, pairs[0].s2, pairs[0].n2 = b"ACGUACGU", 8, b"ACGU", 4
    small = np.zeros(4, dtype=np.float32)
    assert lib.rp_run_dense(stage.ctx, pairs, 1, C.byref(opts), small.ctypes.data, small.size) == 9  # RP_ERR_CAPACITY
    assert lib.rp_run_dense(stage.ctx, None, 1, C.byref(opts), small.ctypes.data, small.size) == 1
    assert stage.run_dense([], opts) == []
    with pytest.raises(RpError):
        stage.run_dense([("", "ACGU")], opts)


@pytest.mark.parametrize("n1,n2", [(95, 1), (96, 3), (60, 40), (150, 65), (107, 108), (108, 108), (215, 1), (111, 112), (112, 112), (223, 1), (224, 2)])
def test_kernel_class_boundaries(stage, oracle, lib, n1, n2):
    """Lengths around the routing boundaries of rp_kernel_plan (two band CTAs per SM / one / general
    kernel): every route gives the oracle's numbers."""
    from ractip_b200 import default_opts
    rng = np.random.default_rng(31 * n1 + n2)
    opts = default_opts()
    s1, s2 = rand_seq(rng, n1), rand_seq(rng, n2)
    routes = {lib.rp_kernel_plan(n, 0, None) for n in (n1, n2, n1 + n2)}
    assert routes <= {0, 1, 2, 3}
    r = stage.run_dense([(s1, s2)], opts)[0]
    _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, f"{n1}x{n2} routes {sorted(routes)}")


def test_band_and_general_kernels_agree(model, bundled, monkeypatch):
    """The shared-memory band kernel and the HBM-table general kernel compute the same matrices
    (RP_BAND=0 routes everything to the general kernel: A/B aid)."""
    from ractip_b200 import ProbabilityStage, default_opts, zscore_shuffles
    s1, s2 = bundled["sequences"]["MicA"], bundled["sequences"]["ompA"]
    r1, r2 = zscore_shuffles(s1, s2, 6, 1)
    pairs = list(zip(r1, r2)) + [(bundled["sequences"]["CopA"], bundled["sequences"]["CopT"])]
    opts = default_opts()
    st_band = ProbabilityStage(model)
    a = st_band.run_dense(pairs, opts)
    st_band.close()
    monkeypatch.setenv("RP_BAND", "0")
    st_gen = ProbabilityStage(model)
    b = st_gen.run_dense(pairs, opts)
    st_gen.close()
    for x, y in zip(a, b):
        for name in ("bp1", "bp2", "up1", "up2"):
            assert np.abs(getattr(x, name).astype(np.float64) - getattr(y, name)).max() <= TOL, name
        both = (x.hp != 0) & (y.hp != 0)
        assert np.abs(x.hp[both].astype(np.float64) - y.hp[both]).max() <= TOL
        mism = (x.hp != 0) != (y.hp != 0)
        if mism.any():
            assert _near_threshold(np.where(x.hp != 0, x.hp, y.hp)[mism], opts.th_hy).all()


@pytest.mark.parametrize("wide", [10])
def test_wide_split_sum_bands(model, oracle, monkeypatch, wide):
    """Long-problem schedule of the general kernel (128-register build, split sums in bands of `wide`
    diagonals: far pass + near terms at the finish), forced onto mid-size problems the oracle does quickly."""
    from ractip_b200 import ProbabilityStage, default_opts
    monkeypatch.setenv("RP_MCC_LONG_N", "216")
    rng = np.random.default_rng(4100 + wide)
    opts = default_opts()
    pairs = [(rand_seq(rng, 300), rand_seq(rng, 130)), (rand_seq(rng, 217), rand_seq(rng, 260))]
    st = ProbabilityStage(model)
    try:
        for (s1, s2), r in zip(pairs, st.run_dense(pairs, opts)):
            _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, f"wide={wide} {len(s1)}x{len(s2)}")
    finally:
        st.close()


def test_long_pair_default_routing(stage, oracle):
    """620 x 300 nt: the two-strand problem (920 nt) takes the wide-band build by default, the single
    strands the 64-register build."""
    from ractip_b200 import default_opts
    rng = np.random.default_rng(920)
    s1, s2 = rand_seq(rng, 620), rand_seq(rng, 300)
    opts = default_opts()
    r = stage.run_dense([(s1, s2)], opts)[0]
    _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, "620x300")


def test_pinned_host_buffer_is_written_in_place(stage, bundled):
    """rp_run_dense into a page-locked buffer and into pageable memory give the same bytes."""
    from ractip_b200 import default_opts
    seqs = bundled["sequences"]
    pairs = [(seqs["DIS"], seqs["DIS"]), (seqs["MicA"], seqs["ompA"]), (seqs["CopA"], seqs["CopT"])]
    for duplex in (0, 1):
        opts = default_opts()
        opts.use_pf_duplex = duplex
        a = stage.run_dense(pairs, opts)
        b = stage.run_dense(pairs, opts, pinned=True)
        for x, y in zip(a, b):
            for name in ("bp1", "bp2", "up1", "up2", "hp"):
                assert np.array_equal(getattr(x, name), getattr(y, name)), (duplex, name)


@pytest.mark.parametrize("cluster", [None, "0"])
def test_configs4_size_pair_matches_oracle(model, oracle, monkeypatch, cluster):
    """One pair of BASELINE configs[4]'s size (1000 x 500 nt, two-strand problem of 1500 nt) against the oracle:
    on the default route for a single pair (16-CTA clusters) and on the batch's route (one CTA per problem,
    wide bands; RP_CLUSTER=0)."""
    from ractip_b200 import ProbabilityStage, default_opts
    if cluster is not None:
        monkeypatch.setenv("RP_CLUSTER", cluster)
    rng = np.random.default_rng(20261018)
    s1 = "".join("ACGU"[x] for x in rng.integers(0, 4, 1000))
    s2 = "".join("ACGU"[x] for x in rng.integers(0, 4, 500))
    opts = default_opts()
    st = ProbabilityStage(model)
    try:
        r = st.run_dense([(s1, s2)], opts, pinned=True)[0]
    finally:
        st.close()
    _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, "1000x500")


@pytest.mark.parametrize("n1,n2,seed", [(745, 31, 5), (513, 512, 6), (700, 333, 7)])
def test_long_ragged_pairs_match_oracle(model, oracle, monkeypatch, n1, n2, seed):
    """The long-problem build (wide split-sum bands, staged interior tiles, row-major copies) on shapes that put
    the chunk and strand-segment boundaries in odd places: a nick 31 nt from the 3' end, diagonals one cell longer than
    the CTA width, a strand-2 segment shorter than a chunk.  RP_CLUSTER=0 keeps the batch's route (one CTA per problem)."""
    from ractip_b200 import ProbabilityStage, default_opts
    monkeypatch.setenv("RP_CLUSTER", "0")
    monkeypatch.setenv("RP_MCC_LONG_N", "500")   # the 513-nt strands take the long build too
    rng = np.random.default_rng(seed)
    s1 = "".join("ACGU"[x] for x in rng.integers(0, 4, n1))
    s2 = "".join("ACGU"[x] for x in rng.integers(0, 4, n2))
    opts = default_opts()
    st = ProbabilityStage(model)
    try:
        r = st.run_dense([(s1, s2)], opts, pinned=True)[0]
    finally:
        st.close()
    _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, f"{n1}x{n2}")


def test_split_fetch_of_uniform_batches(stage, model, bundled, monkeypatch):
    """Shuffle batches (every pair the same lengths) whose problems fall into both band classes are fetched in
    two parts -- the long class's sections while the short class still runs -- and give the same bytes as the
    single copy (RP_NO_SPLIT_FETCH=1)."""
    from ractip_b200 import ProbabilityStage, default_opts, zscore_shuffles
    s1, s2 = bundled["sequences"]["MicA"], bundled["sequences"]["ompA"]
    r1, r2 = zscore_shuffles(s1, s2, 12, 3)
    pairs = list(zip(r1, r2))
    opts = default_opts()
    a = stage.run_dense(pairs, opts)
    b = stage.run_dense(pairs, opts, pinned=True)
    monkeypatch.setenv("RP_NO_SPLIT_FETCH", "1")   # read when a context is created
    st = ProbabilityStage(model)
    try:
        c = st.run_dense(pairs, opts)
    finally:
        st.close()
    for x, y, z in zip(a, b, c):
        for name in ("bp1", "bp2", "up1", "up2", "hp"):
            assert np.array_equal(getattr(x, name), getattr(z, name)), name
            assert np.array_equal(getattr(y, name), getattr(z, name)), name
        assert x.bp2.max() > 0 and x.bp1.max() > 0 and x.up1.max() > 0


@pytest.mark.parametrize("cluster,long_n", [("0", "224"), ("8", "224"), ("16", "224"), ("0", "100000")])
def test_multi_cta_wavefront_matches_oracle(model, oracle, monkeypatch, cluster, long_n):
    """Long problems, few of them: one problem per thread-block cluster (RP_CLUSTER=8 / 16 force the multi-CTA
    wavefront with that cluster size, 0 the one-CTA-per-problem builds: the 128-register wide-band one with
    RP_MCC_LONG_N=224, the 64-register one with the threshold out of reach); all against the oracle, incl.
    unpaired windows and a nick."""
    from ractip_b200 import ProbabilityStage, default_opts
    monkeypatch.setenv("RP_CLUSTER", cluster)
    monkeypatch.setenv("RP_MCC_LONG_N", long_n)
    rng = np.random.default_rng(8800)
    opts = default_opts()
    pairs = [(rand_seq(rng, 300), rand_seq(rng, 130)), (rand_seq(rng, 230), rand_seq(rng, 261)), (rand_seq(rng, 40), rand_seq(rng, 610))]
    st = ProbabilityStage(model)
    try:
        for (s1, s2), r in zip(pairs, st.run_dense(pairs, opts)):
            _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, f"cluster={cluster} {len(s1)}x{len(s2)}")
    finally:
        st.close()


# ---------------------------------------------------------------------------------------------
# round 2: end-to-end consumers, oracle-derived lists, the full batch, non-default models
# ---------------------------------------------------------------------------------------------
def test_joint_structures_identical_to_oracle_on_all_bundled_pairs(stage, oracle, model, bundled):
    """north_star: identical predicted joint dot-bracket structures on every data/*.fa pair.  The integer
    programme (ractip_b200/ip.py over csrc/ipmodel.cpp; src/ractip.cpp:552-1316) is fed once with the GPU's
    matrices, once with the GPU's thresholded lists (x, y, z, v, w) and once with the oracle's matrices."""
    from ractip_b200 import default_opts, solve_joint
    from test_ip import README_DIS, oracle_probs
    opts = default_opts()
    pairs = [(bundled["sequences"][a], bundled["sequences"][b]) for a, b in bundled["pairs"]]
    dense = stage.run_dense(pairs, opts)
    lists = stage.run_sparse(pairs, opts)
    for (a, b), (s1, s2), d, l in zip(bundled["pairs"], pairs, dense, lists):
        g = solve_joint(model, s1, s2, d, energies=True)
        gl = solve_joint(model, s1, s2, d, recs=l)
        o = solve_joint(model, s1, s2, oracle_probs(oracle, s1, s2), energies=True)
        assert (g.r1, g.r2) == (o.r1, o.r2), (a, b)
        assert (gl.r1, gl.r2) == (o.r1, o.r2), (a, b, "lists")
        assert (g.e1, g.e2, g.e3) == (o.e1, o.e2, o.e3)
        assert abs(g.objective - o.objective) < 1e-5
    # the README example (README.md:91-97): exact once the near-threshold window 11..23 is not a variable
    from ractip_b200 import default_ip_opts
    s = bundled["sequences"]["DIS"]
    k = [p for p, (a, b) in enumerate(bundled["pairs"]) if a == "DIS"][0]
    r = solve_joint(model, s, s, dense[k], default_ip_opts(th_ac=0.004))
    assert (r.r1, r.r2) == README_DIS


def test_sparse_lists_against_oracle_derived_lists(stage, oracle, bundled):
    """x, y, z, v, w records of rp_run_sparse against lists cut from the ORACLE's matrices in the reference's
    creation order (src/ractip.cpp:557-567, 578-588, 598-609, 619-628, 639-648)."""
    from ractip_b200 import default_opts
    from test_dist import oracle_lists
    for kw in (dict(), dict(min_w=3, max_w=8, th_ac=0.01), dict(min_w=1, max_w=4), dict(max_w=1, min_w=5)):
        opts = default_opts(**kw)
        pairs = [(bundled["sequences"][a], bundled["sequences"][b]) for a, b in bundled["pairs"]]
        for (s1, s2), sp in zip(pairs, stage.run_sparse(pairs, opts)):
            want = oracle_lists(oracle, s1, s2, opts)
            for got, ref, th in zip((sp.x, sp.y, sp.z, sp.v, sp.w), want,
                                    (opts.th_ss, opts.th_ss, opts.th_hy, opts.th_ac, opts.th_ac)):
                gi = [(int(r["i"]), int(r["j"])) for r in got]
                ri = [(i, j) for i, j, _ in ref]
                if gi != ri:   # only values within float noise of the threshold may differ in presence
                    odd = set(gi) ^ set(ri)
                    pv = {(i, j): p for i, j, p in ref}
                    pv.update({(int(r["i"]), int(r["j"])): float(r["p"]) for r in got})
                    assert all(abs(pv[k] - float(np.float32(th))) < 3e-7 for k in odd), (kw, odd)
                    assert [k for k in gi if k not in odd] == [k for k in ri if k not in odd]
                else:
                    assert np.abs(np.array([r["p"] for r in got], dtype=np.float64) -
                                  np.array([p for _, _, p in ref], dtype=np.float64)).max(initial=0) <= TOL


def test_full_1000_shuffle_batch_against_the_oracle(stage, oracle, bundled):
    """BASELINE configs[3] at full size: EVERY one of the 1000 shuffled pairs against the oracle."""
    from concurrent.futures import ThreadPoolExecutor
    from ractip_b200 import default_opts, zscore_shuffles
    s1, s2 = bundled["sequences"]["MicA"], bundled["sequences"]["ompA"]
    r1, r2 = zscore_shuffles(s1, s2, 1000, 1)
    pairs = list(zip(r1, r2))
    opts = default_opts()
    res = stage.run_dense(pairs, opts)
    with ThreadPoolExecutor(16) as ex:   # the oracle releases the GIL inside its C calls
        oras = list(ex.map(lambda p: _oracle_pair(oracle, p[0], p[1], opts), pairs))
    for k, ((a, c), r, ora) in enumerate(zip(pairs, res, oras)):
        _compare(r, ora, a, c, opts, f"shuffle {k}")


def test_250_shuffle_batch_against_the_oracle(stage, oracle, bundled):
    """250 shuffled pairs: on a B200 the unpaired-window passes run as jobs of their own inside the band kernel,
    each waiting on its problem's wavefronts.  Every pair against the oracle; bitwise repeatable."""
    from concurrent.futures import ThreadPoolExecutor
    from ractip_b200 import default_opts, zscore_shuffles
    s1, s2 = bundled["sequences"]["MicA"], bundled["sequences"]["ompA"]
    r1, r2 = zscore_shuffles(s1, s2, 250, 1)
    pairs = list(zip(r1, r2))
    opts = default_opts()
    b = stage.batch(pairs, opts)
    b.run()
    flat = b.fetch_dense().copy()
    b.run()
    assert np.array_equal(flat, b.fetch_dense()), "the 250-pair batch is not bitwise repeatable"
    res = b.split_dense(flat)
    b.close()
    with ThreadPoolExecutor(16) as ex:   # the oracle releases the GIL inside its C calls
        oras = list(ex.map(lambda p: _oracle_pair(oracle, p[0], p[1], opts), pairs))
    for k, ((a, c), r, ora) in enumerate(zip(pairs, res, oras)):
        _compare(r, ora, a, c, opts, f"shuffle {k}")


@pytest.mark.parametrize("variant", ["special_hp0", "pf_smooth0", "par_overlay"])
def test_parity_under_non_default_models(variant, bundled, tmp_path):
    """The kernels under other energy models: tetra_loop off, pf_smooth off, and a -P overlay
    (rp_model_read_par, src/ractip.cpp:1568-1569) that changes stacking, hairpin and multiloop values."""
    from oracle.oracle import Oracle
    from ractip_b200 import ProbabilityStage, default_model, default_opts
    m = default_model()
    if variant == "special_hp0":
        m.special_hp = 0
    elif variant == "pf_smooth0":
        m.pf_smooth = 0
    else:
        par = tmp_path / "overlay.par"
        lines = ["## RNAfold parameter file v2.0", "", "# stack"]
        rng = np.random.default_rng(5)
        for _ in range(7):
            lines.append(" ".join(str(int(v)) for v in rng.integers(-340, -60, 7)))
        lines += ["", "# hairpin", "INF INF INF 540 560 570 540 600 550 640",
                  "650 660 670 680 690 690 700 710 710 720", "720 730 730 740 740 750 750 750 760 760", "770",
                  "", "# ML_params", "0 0 930 3000 -90 -220", "", "# NINIO", "60 320 300", "", "#END", ""]
        par.write_text("\n".join(lines))
        m = default_model(param_file=str(par))
        assert m.ML_closing37 == 930 and m.ninio37 == 60
    st = ProbabilityStage(m)
    orc = Oracle(m)
    opts = default_opts()
    try:
        for a, b in [("DIS", "DIS"), ("CopA", "CopT"), ("MicA", "ompA")]:
            s1, s2 = bundled["sequences"][a], bundled["sequences"][b]
            _compare(st.solve_probabilities(s1, s2, opts), _oracle_pair(orc, s1, s2, opts), s1, s2, opts, variant)
    finally:
        st.close()


def test_random_sweep_of_lengths_nick_positions_and_letters(stage, oracle):
    """Hypothesis-style sweep: lengths 1..260 (every kernel route), every nick position class, N / T /
    lower-case letters; 120 seeded pairs in three ragged batches."""
    from ractip_b200 import default_opts
    rng = np.random.default_rng(20261018)
    opts = default_opts()
    alphabets = ["ACGU", "ACGU", "GCGCAU", "ACGUN", "ACGTacgu"]
    for batch in range(3):
        pairs = []
        for _ in range(40):
            tot = int(rng.choice([rng.integers(2, 40), rng.integers(40, 120), rng.integers(120, 261)]))
            n1 = int(rng.integers(1, tot))
            al = alphabets[int(rng.integers(0, len(alphabets)))]
            pairs.append((rand_seq(rng, n1, al), rand_seq(rng, tot - n1, al)))
        for (s1, s2), r in zip(pairs, stage.run_dense(pairs, opts)):
            _compare(r, _oracle_pair(oracle, s1, s2, opts), s1, s2, opts, f"sweep {len(s1)}x{len(s2)}")


def test_single_sequence_request_and_context_lifetime(oracle, model, bundled):
    """A pair with an empty second sequence computes s1's sections only (RactIP::rnafold on its own,
    src/ractip.cpp:308-382); closing the stage while a batch is alive is safe (the last batch tears it down)."""
    from ractip_b200 import ProbabilityStage, default_opts
    st = ProbabilityStage(model)
    s = bundled["sequences"]["MicA"]
    bp, off, up = st.rnafold(s, 15)
    obp, oup = oracle.rnafold(s, 15)
    assert np.abs(bp.astype(np.float64) - obp).max() <= TOL and np.abs(up.astype(np.float64) - oup).max() <= TOL
    assert 1 <= st.last_timing().kernel_launches <= 2   # the band kernel (+ the deferred unpaired-window kernel)
    mixed = st.run_dense([(s, ""), (bundled["sequences"]["DIS"], bundled["sequences"]["DIS"])], default_opts())
    assert mixed[0].hp.shape == (len(s) + 1, 1) and not mixed[0].hp.any() and mixed[0].up2.shape == (0, 15)
    assert np.abs(mixed[0].bp1.astype(np.float64) - obp).max() <= TOL
    assert mixed[1].hp.max() > 0.9
    b = st.batch([(s, s)], default_opts())
    b.run()
    st.close()          # the context stays alive underneath until its last batch goes
    flat = b.fetch_dense()
    assert np.abs(b.split_dense(flat)[0].bp1.astype(np.float64) - obp).max() <= TOL
    b.close()
