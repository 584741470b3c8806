"""The batch's probability matrices handed to PyTorch as CUDA tensors: the packed dense block
(rp_batch_dense_device, DeviceBatch.dense_tensor) and the padded square tensors (rp_square_plan,
rp_batch_square_device, DeviceBatch.tensors).

Host-side tests pin the square layout and a numpy expansion of the packed layout; the GPU tests
require the device results to equal, bit for bit, fetch_dense() and that expansion of it."""
import ctypes as C

import numpy as np
import pytest

from conftest import rand_seq

KEYS = ("bp1", "bp2", "up1", "up2", "hp")


def _pairs_array(lens):
    """rp_pair array with the given lengths; the plans read lengths only, so every sequence is one short buffer."""
    from ractip_b200._lib import RpPair
    arr = (RpPair * max(len(lens), 1))()
    buf = C.create_string_buffer(b"A" * 16)
    for k, (n1, n2) in enumerate(lens):
        arr[k].s1, arr[k].n1 = C.cast(buf, C.c_char_p), n1
        arr[k].s2, arr[k].n2 = (C.cast(buf, C.c_char_p) if n2 else None), n2
    return arr, buf


def _square_plan(lib, lens, opts):
    from ractip_b200._lib import RpSquareLayout
    arr, keep = _pairs_array(lens)
    lay = RpSquareLayout()
    rc = lib.rp_square_plan(arr, len(lens), C.byref(opts), C.byref(lay))
    return rc, lay


def _dense_layouts(lib, lens, opts):
    from ractip_b200._lib import RpDenseLayout
    arr, keep = _pairs_array(lens)
    lay = (RpDenseLayout * max(len(lens), 1))()
    tot = C.c_size_t()
    assert lib.rp_dense_plan(arr, len(lens), C.byref(opts), lay, C.byref(tot)) == 0
    return lay, tot.value


def square_reference(flat, layouts, lens, W):
    """numpy expansion of the packed layout (rp_dense_plan) into the square tensors of rp_square_plan."""
    from ractip_b200 import bp_offsets
    B = len(lens)
    N1 = max((a for a, _ in lens), default=0)
    N2 = max((b for _, b in lens), default=0)
    out = {"bp1": np.zeros((B, N1 + 1, N1 + 1), np.float32), "bp2": np.zeros((B, N2 + 1, N2 + 1), np.float32),
           "up1": np.zeros((B, N1, W), np.float32), "up2": np.zeros((B, N2, W), np.float32),
           "hp": np.zeros((B, N1 + 1, N2 + 1), np.float32)}
    for k, (n1, n2) in enumerate(lens):
        L = layouts[k]
        for key, n, off in (("bp1", n1, L.bp1), ("bp2", n2, L.bp2)):
            i, j = np.triu_indices(n + 1, 1)
            keep = i >= 1                    # bp[offset[i]+j], 1 <= i < j <= n
            i, j = i[keep], j[keep]
            v = flat[off + bp_offsets(n)[i].astype(np.int64) + j]
            out[key][k, i, j] = v
            out[key][k, j, i] = v
        out["up1"][k, :n1] = flat[L.up1:L.up1 + n1 * W].reshape(n1, W)
        out["up2"][k, :n2] = flat[L.up2:L.up2 + n2 * W].reshape(n2, W)
        if n2:
            out["hp"][k, :n1 + 1, :n2 + 1] = flat[L.hp:L.hp + L.n_hp].reshape(n1 + 1, n2 + 1)
    return out


# ------------------------------------------------------------------------------------------- host only
@pytest.mark.parametrize("max_w", [0, 1, 15])
def test_square_plan_shapes(lib, max_w):
    from ractip_b200 import default_opts
    o = default_opts(max_w=max_w)
    lens = [(10, 9), (72, 137), (5, 0), (130, 31)]
    rc, s = _square_plan(lib, lens, o)
    assert rc == 0
    assert (s.B, s.N1, s.N2, s.W) == (4, 130, 137, max_w)
    assert (s.n_bp1, s.n_bp2, s.n_up1, s.n_up2, s.n_hp) == (
        4 * 131 * 131, 4 * 138 * 138, 4 * 130 * max_w, 4 * 137 * max_w, 4 * 131 * 138)
    # every second sequence empty: N2 = 0, bp2 is one zero per pair, up2 has no rows
    rc, s = _square_plan(lib, [(7, 0), (3, 0)], o)
    assert rc == 0 and (s.B, s.N1, s.N2) == (2, 7, 0)
    assert (s.n_bp1, s.n_bp2, s.n_up1, s.n_up2, s.n_hp) == (2 * 64, 2, 2 * 7 * max_w, 0, 2 * 8)
    rc, s = _square_plan(lib, [], o)
    assert rc == 0 and (s.B, s.n_bp1, s.n_hp) == (0, 0, 0)


def test_square_plan_negative_max_w_is_no_window(lib):
    from ractip_b200 import default_opts
    rc, s = _square_plan(lib, [(4, 6)], default_opts(max_w=-3))
    assert rc == 0 and s.W == 0 and s.n_up1 == 0 and s.n_up2 == 0


def test_square_plan_rejects_overflow_and_bad_arguments(lib):
    from ractip_b200 import default_opts
    o = default_opts()
    big = 2 ** 31 - 1
    assert _square_plan(lib, [(2 ** 20, 2 ** 20)], o)[0] == 0
    assert _square_plan(lib, [(big, 1)] * 4, o)[0] == 1        # 4 * 2^62 elements
    assert _square_plan(lib, [(big, big)], o)[0] == 1          # 2^62 elements fit, their bytes do not
    assert _square_plan(lib, [(1, 1), (1, big)] * 2, o)[0] == 1
    assert _square_plan(lib, [(0, 3)], o)[0] == 1              # n1 must be >= 1
    arr, keep = _pairs_array([(3, 3)])
    from ractip_b200._lib import RpSquareLayout
    lay = RpSquareLayout()
    assert lib.rp_square_plan(None, 1, C.byref(o), C.byref(lay)) == 1
    assert lib.rp_square_plan(arr, 1, None, C.byref(lay)) == 1
    assert lib.rp_square_plan(arr, 1, C.byref(o), None) == 1
    assert lib.rp_square_plan(arr, -1, C.byref(o), C.byref(lay)) == 1


def test_device_exits_reject_a_null_batch(lib):
    assert lib.rp_batch_dense_device(None, None, 0) == 1
    assert lib.rp_batch_square_device(None, None, None, None, None, None) == 1
    assert lib.rp_get_stream(None, None) == 1


def test_reference_expansion_of_hand_built_layouts(lib):
    """Two pairs, (3, 2) and (1, 0), max_w 2, every packed float numbered 1, 2, 3, ... in buffer order."""
    from ractip_b200 import default_opts
    lens = [(3, 2), (1, 0)]
    lay, tot = _dense_layouts(lib, lens, default_opts(max_w=2))
    # pair 0: bp1 10 floats, bp2 6, up1 6, up2 4, hp 12 = 38; pair 1: bp1 3, bp2 1, up1 2, up2 0, hp 2 = 8
    assert tot == 46 and lay[1].bp1 == 38
    flat = np.arange(1, tot + 1, dtype=np.float32)
    sq = square_reference(flat, lay, lens, 2)
    # L = 3: offset = [0, 3, 5, 6]; (1,2) -> 5, (1,3) -> 6, (2,3) -> 8 (0-based), so values 6, 7, 9
    np.testing.assert_array_equal(sq["bp1"][0], [[0, 0, 0, 0], [0, 0, 6, 7], [0, 6, 0, 9], [0, 7, 9, 0]])
    # L = 2 starting at 10: offset = [0, 2, 3]; (1,2) -> 10 + 4 -> value 15
    np.testing.assert_array_equal(sq["bp2"][0], [[0, 0, 0], [0, 0, 15], [0, 15, 0]])
    np.testing.assert_array_equal(sq["up1"][0], [[17, 18], [19, 20], [21, 22]])
    np.testing.assert_array_equal(sq["up2"][0], [[23, 24], [25, 26]])
    np.testing.assert_array_equal(sq["hp"][0], np.arange(27, 39).reshape(4, 3))
    # pair 1: L = 1 has no pair (1 <= i < j <= 1), a lone sequence has zero bp2 / up2 / hp, rows past n1 are 0
    np.testing.assert_array_equal(sq["bp1"][1], np.zeros((4, 4)))
    np.testing.assert_array_equal(sq["bp2"][1], np.zeros((3, 3)))
    np.testing.assert_array_equal(sq["up1"][1], [[43, 44], [0, 0], [0, 0]])
    np.testing.assert_array_equal(sq["up2"][1], np.zeros((2, 2)))
    np.testing.assert_array_equal(sq["hp"][1], np.zeros((4, 3)))


def test_reference_expansion_matches_per_pair_indexing(lib):
    """The expansion against the reference's own indexing, bp[offset[i]+j] and hp[i][j], on a ragged batch."""
    from ractip_b200 import bp_offsets, default_opts
    lens = [(6, 4), (2, 7), (9, 0)]
    W = 3
    lay, tot = _dense_layouts(lib, lens, default_opts(max_w=W))
    flat = np.random.default_rng(5).random(tot, dtype=np.float32)
    sq = square_reference(flat, lay, lens, W)
    for k, (n1, n2) in enumerate(lens):
        L = lay[k]
        for key, n, off in (("bp1", n1, L.bp1), ("bp2", n2, L.bp2)):
            o = bp_offsets(n)
            P = sq[key][k]
            assert (P == P.T).all()
            for i in range(P.shape[0]):
                for j in range(P.shape[1]):
                    want = flat[off + o[i] + j] if 1 <= i < j <= n else (flat[off + o[j] + i] if 1 <= j < i <= n else 0)
                    assert P[i, j] == want, (key, k, i, j)
        hp = flat[L.hp:L.hp + L.n_hp].reshape(n1 + 1, n2 + 1) if n2 else np.zeros((n1 + 1, 1), np.float32)
        assert (sq["hp"][k, :n1 + 1, :n2 + 1] == hp[:, :n2 + 1]).all() and not sq["hp"][k, n1 + 1:].any()
        assert not sq["hp"][k, :, n2 + 1:].any()


# ------------------------------------------------------------------------------------------------- GPU
def _case(name, bundled):
    from ractip_b200 import default_opts
    seqs = bundled["sequences"]
    if name == "bundled":
        return [(seqs[a], seqs[b]) for a, b in bundled["pairs"]], default_opts()
    if name == "edge":   # the lengths of test_gpu_parity.py::test_edge_and_ragged_lengths, as one ragged batch
        rng = np.random.default_rng(31)
        lens = [(1, 1), (2, 5), (4, 4), (5, 5), (7, 3), (9, 12), (33, 64), (130, 31)]
        return [(rand_seq(rng, a), rand_seq(rng, b)) for a, b in lens], default_opts()
    if name == "single":   # a lone sequence (n2 == 0) next to an ordinary pair
        return [(seqs["MicA"], ""), (seqs["DIS"], seqs["DIS"])], default_opts()
    if name == "duplex":   # --duplex: dense hp
        return [(seqs["DIS"], seqs["DIS"]), (seqs["MicA"], seqs["ompA"]), ("GGGAAACC", "GGUUUCCC"), ("A", "U")], \
            default_opts(use_pf_duplex=1)
    if name == "long":   # one pair of BASELINE configs[4]'s size
        rng = np.random.default_rng(20261018)
        return [(rand_seq(rng, 1000), rand_seq(rng, 500))], default_opts()
    raise KeyError(name)


CASES = ["bundled", "edge", "single", "duplex", "long"]


@pytest.fixture(scope="module", params=CASES)
def ran(request, stage, bundled):
    """A batch of the case, run, with its fetch_dense() block and the numpy expansion of that block."""
    pairs, opts = _case(request.param, bundled)
    b = stage.batch(pairs, opts)
    b.run()
    flat = b.fetch_dense()[:b.total_floats]
    lens = [(len(s1), len(s2)) for s1, s2 in pairs]
    ref = square_reference(flat, b.layout, lens, max(opts.max_w, 0))
    yield b, flat, ref
    b.close()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _assert_square(got, ref, lens, stage):
    import torch
    for k in KEYS:
        t = got[k]
        assert t.dtype == torch.float32 and t.device == torch.device("cuda", stage.device) and t.is_contiguous()
        assert tuple(t.shape) == ref[k].shape, k
        assert np.array_equal(_bits(t.cpu().numpy()), _bits(ref[k])), k
    assert got["n1"].dtype == torch.int32 and got["n1"].cpu().tolist() == [a for a, _ in lens]
    assert got["n2"].dtype == torch.int32 and got["n2"].cpu().tolist() == [b for _, b in lens]


@pytest.mark.gpu
def test_dense_tensor_is_bitwise_fetch_dense(ran):
    b, flat, ref = ran
    t = b.dense_tensor()
    assert t.numel() == b.total_floats
    assert np.array_equal(_bits(t.cpu().numpy()), _bits(flat))


@pytest.mark.gpu
def test_square_tensors_are_bitwise_the_expansion_of_fetch_dense(ran, stage):
    b, flat, ref = ran
    _assert_square(b.tensors(), ref, [(len(s1), len(s2)) for s1, s2 in b.pairs], stage)


@pytest.mark.gpu
def test_kernel_writes_its_own_padding(ran, stage):
    """Output buffers pre-filled with NaN: every element of the square tensors is written; the dense copy
    writes exactly total_floats floats."""
    import torch
    b, flat, ref = ran
    lay = b.square_layout()
    shapes = {"bp1": (lay.B, lay.N1 + 1, lay.N1 + 1), "bp2": (lay.B, lay.N2 + 1, lay.N2 + 1),
              "up1": (lay.B, lay.N1, lay.W), "up2": (lay.B, lay.N2, lay.W), "hp": (lay.B, lay.N1 + 1, lay.N2 + 1)}
    dev = stage.torch_device()
    out = {k: torch.full(shapes[k], float("nan"), dtype=torch.float32, device=dev) for k in KEYS}
    dense = torch.full((b.total_floats + 64,), float("nan"), dtype=torch.float32, device=dev)
    with stage._torch_stream():
        ptrs = [C.c_void_p(out[k].data_ptr() if out[k].numel() else None) for k in KEYS]
        assert b.lib.rp_batch_square_device(b.handle, *ptrs) == 0
        assert b.lib.rp_batch_dense_device(b.handle, C.c_void_p(dense.data_ptr()), dense.numel()) == 0
    for k in KEYS:
        assert np.array_equal(_bits(out[k].cpu().numpy()), _bits(ref[k])), k
    d = dense.cpu().numpy()
    assert np.array_equal(_bits(d[:b.total_floats]), _bits(flat)) and np.isnan(d[b.total_floats:]).all()
    # NULL skips a tensor and leaves its buffer alone
    out["hp"].fill_(float("nan"))
    with stage._torch_stream():
        assert b.lib.rp_batch_square_device(b.handle, None, None, None, None, None) == 0
        assert b.lib.rp_batch_square_device(b.handle, C.c_void_p(out["bp1"].data_ptr()), None, None, None, None) == 0
    assert np.isnan(out["hp"].cpu().numpy()).all()
    assert np.array_equal(_bits(out["bp1"].cpu().numpy()), _bits(ref["bp1"]))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_consumed_by_torch_on_a_side_stream_without_synchronise(stage, bundled, case):
    """A fresh batch runs on the context's own stream; its tensors are taken and consumed by torch ops on another
    stream while the kernels may still be running.  The device-side wait orders them: the consumers see the final
    values (checked after the fact against fetch_dense())."""
    import torch
    pairs, opts = _case(case, bundled)
    lens = [(len(s1), len(s2)) for s1, s2 in pairs]
    b = stage.batch(pairs, opts)
    try:
        side = torch.cuda.Stream(stage.torch_device())
        b.run()
        with torch.cuda.stream(side):
            t = b.tensors()
            d = b.dense_tensor()
            consumed = {k: t[k] * 1.0 for k in KEYS}   # torch ops on the same stream, no synchronise
            consumed["n1"], consumed["n2"] = t["n1"] + 0, t["n2"] + 0
            dsum = (d * 1.0).clone()
        side.synchronize()
        flat = b.fetch_dense()[:b.total_floats]
        assert np.array_equal(_bits(dsum.cpu().numpy()), _bits(flat))
        _assert_square(consumed, square_reference(flat, b.layout, lens, max(opts.max_w, 0)), lens, stage)
    finally:
        b.close()
    # the context is back on its own stream
    ptr = C.c_void_p()
    assert stage.lib.rp_get_stream(stage.ctx, C.byref(ptr)) == 0
    assert ptr.value and ptr.value != side.cuda_stream


@pytest.mark.gpu
def test_run_tensors_and_documented_errors(stage, bundled):
    import torch
    pairs, opts = _case("bundled", bundled)
    lens = [(len(s1), len(s2)) for s1, s2 in pairs]
    t = stage.run_tensors(pairs, opts)
    b = stage.batch(pairs, opts)
    try:
        b.run()
        flat = b.fetch_dense()[:b.total_floats]
        _assert_square(t, square_reference(flat, b.layout, lens, opts.max_w), lens, stage)
        buf = torch.empty(b.total_floats, dtype=torch.float32, device=stage.torch_device())
        lib = b.lib
        assert lib.rp_batch_dense_device(b.handle, C.c_void_p(buf.data_ptr()), b.total_floats - 1) == 9   # capacity
        assert lib.rp_batch_dense_device(b.handle, None, b.total_floats) == 1                             # NULL
        assert lib.rp_batch_square_device(None, C.c_void_p(buf.data_ptr()), None, None, None, None) == 1
    finally:
        b.close()
    # an empty batch: no-ops, empty tensors
    e = stage.batch([], opts)
    try:
        e.run()
        assert e.dense_tensor().numel() == 0
        te = e.tensors()
        assert all(te[k].numel() == 0 for k in KEYS) and te["n1"].numel() == 0
        buf = torch.empty(1, dtype=torch.float32, device=stage.torch_device())
        assert e.lib.rp_batch_dense_device(e.handle, C.c_void_p(buf.data_ptr()), 0) == 0
    finally:
        e.close()
