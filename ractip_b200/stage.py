"""Host-side mirror of RactIP's probability stage over the C ABI.

`ProbabilityStage.solve_probabilities(fa1, fa2)` is the three calls
RactIP::solve makes at reference src/ractip.cpp:546-548, returning the same
members it fills (`bp1_, offset1_, up1_, bp2_, offset2_, up2_, hp_`,
src/ractip.cpp:185-191) with the same indexing:

    bp[offset[i] + j]   1-based i<j, offset[i] = i*(2L+1-i)/2   (:316-317,365-367)
    up[i][d]            0-based start i, window i..i+d           (:370-375)
    hp[i][j]            1-based both                             (:404-405,451-453)

All arithmetic runs in the CUDA library; torch/numpy are only used for buffers.
"""
from __future__ import annotations

import contextlib
import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import (RpConstraint, RpDenseLayout, RpModel, RpOpts, RpPair, RpRec, RpSampleLayout, RpSampleOpts,
                   RpSparseCounts, RpSparseLayout, RpSquareLayout, RpStackEnergy, RpTiming,
                   RpUnpairedEnergy)


class RpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"ractip_prob error {code}: {msg}")
        self.code = code


def default_model(use_bl: bool = True, param_file: Optional[str] = None) -> RpModel:
    """Energy tables as RactIP::run primes them (src/ractip.cpp:1566-1569):
    ViennaRNA defaults, then BL* unless --no-bl, then the -P file."""
    lib = _lib.load()
    m = RpModel()
    rc = lib.rp_model_default(C.byref(m), 1 if use_bl else 0)
    if rc and not (rc == 6 and param_file):  # RP_ERR_NO_DEFAULTS is recoverable by a full -P file
        raise RpError(rc, lib.rp_strerror(rc).decode())
    if param_file:
        rc = lib.rp_model_read_par(C.byref(m), param_file.encode())
        if rc:
            raise RpError(rc, lib.rp_strerror(rc).decode())
    return m


def default_opts(**kw) -> RpOpts:
    lib = _lib.load()
    o = RpOpts()
    lib.rp_opts_default(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise TypeError(f"unknown option {k}")
        setattr(o, k, v)
    return o


def bp_offsets(L: int) -> np.ndarray:
    """offset[i] = i*((L+1)+(L+1)-i-1)/2  (src/ractip.cpp:316-317)"""
    i = np.arange(L + 1, dtype=np.int64)
    return (i * ((L + 1) + (L + 1) - i - 1) // 2).astype(np.int32)


@dataclass
class PairProbabilities:
    """What RactIP::solve holds after src/ractip.cpp:546-548."""
    bp1: np.ndarray      # float32 [(L1+1)(L1+2)/2]
    offset1: np.ndarray  # int32 [L1+1]
    up1: np.ndarray      # float32 [L1, max_w]
    bp2: np.ndarray
    offset2: np.ndarray
    up2: np.ndarray
    hp: np.ndarray       # float32 [L1+1, L2+1]


@dataclass
class PairRecords:
    """Thresholded variable lists in the reference's creation order
    (src/ractip.cpp:557-567, 578-588, 598-609) plus the dense window tables."""
    x: np.ndarray   # structured (i, j, p), 0-based, bp1 > th_ss
    y: np.ndarray   # bp2 > th_ss
    z: np.ndarray   # hp > th_hy
    up1: Optional[np.ndarray]   # dense window tables (None when not fetched)
    up2: Optional[np.ndarray]
    v: Optional[np.ndarray] = None   # (start i, length index j, p): up1[i][j] > th_ac, j in [min_w-1, max_w)  (:619-628)
    w: Optional[np.ndarray] = None   # the same for s2 (:639-648)


REC_DTYPE = np.dtype([("i", np.int32), ("j", np.int32), ("p", np.float32)])

# the tensors of DeviceBatch.tensors(), in the argument order of rp_batch_square_device
SQUARE_KEYS = ("bp1", "bp2", "up1", "up2", "hp")
# cudaStreamLegacy: torch's default stream has handle 0, which rp_set_stream reads as "the context's own stream"
_CUDA_STREAM_LEGACY = 1


def _make_pairs(pairs: Sequence[Tuple[str, str]]):
    n = len(pairs)
    arr = (RpPair * max(n, 1))()
    keep = []
    for k, (s1, s2) in enumerate(pairs):
        b1, b2 = s1.encode(), s2.encode()
        keep.append((b1, b2))
        arr[k].s1, arr[k].n1, arr[k].s2, arr[k].n2 = b1, len(b1), b2, len(b2)
    return arr, keep


def _make_constraints(constraints: Sequence[Optional[Tuple[Optional[str], Optional[str]]]], n: int):
    if len(constraints) != n:
        raise ValueError(f"constraints: {len(constraints)} entries for {n} pairs")
    arr = (RpConstraint * max(n, 1))()
    keep = []
    for k, con in enumerate(constraints):
        c1, c2 = con if con is not None else (None, None)
        b1, b2 = (c.encode() if c is not None else None for c in (c1, c2))
        keep.append((b1, b2))
        arr[k].c1, arr[k].c2 = b1, b2
    return arr, keep


def _make_energies(energies, pairs: Sequence[Tuple[str, str]], struct=RpStackEnergy, what="stack_energies",
                   field="e"):
    """one `struct` (rp_stack_energy or rp_unpaired_energy) per pair from (v1, v2) per-base arrays, either None"""
    n = len(pairs)
    if len(energies) != n:
        raise ValueError(f"{what}: {len(energies)} entries for {n} pairs")
    arr = (struct * max(n, 1))()
    keep = []
    for k, (ent, seqs) in enumerate(zip(energies, pairs)):
        for s, (e, seq) in enumerate(zip(ent if ent is not None else (None, None), seqs)):
            if e is None:
                continue
            a = np.ascontiguousarray(e, dtype=np.float64)
            if a.shape != (len(seq),):
                raise ValueError(f"{what}: pair {k}, {field}{s + 1} has shape {a.shape} for {len(seq)} nt")
            keep.append(a)
            setattr(arr[k], f"{field}{s + 1}", a.ctypes.data)
    return arr, keep


def _make_stack_energies(stack_energies, pairs: Sequence[Tuple[str, str]]):
    return _make_energies(stack_energies, pairs)


def shape_deigan(reactivities, slope: float = 1.8, intercept: float = -0.6) -> np.ndarray:
    """Stacking pseudo-energies (kcal/mol) from probing reactivities by Deigan et al.'s rule (rp_shape_deigan):
    slope * ln(r + 1) + intercept for r >= 0, 0 for a missing value (r < 0 or NaN).  The defaults are RNAfold's
    --shapeMethod=D."""
    r = np.ascontiguousarray(reactivities, dtype=np.float64).reshape(-1)
    e = np.empty_like(r)
    rc = _lib.load().rp_shape_deigan(r.ctypes.data, r.size, slope, intercept, e.ctypes.data)
    if rc:
        raise RpError(rc, "rp_shape_deigan")
    return e


# problem names of sample_problems= and the keys of fetch_samples() / sample_tensors(), with their RP_SAMPLE_* bits
SAMPLE_BITS = {"s1": 1, "s2": 2, "co": 4}


def sample_opts(num: int, seed: int = 1, problems: Sequence[str] = ("s1", "s2", "co")) -> RpSampleOpts:
    """rp_sample_opts: `num` samples of each of `problems` ("s1", "s2", "co"), drawn with `seed`."""
    bits = 0
    for name in problems:
        if name not in SAMPLE_BITS:
            raise ValueError(f"sample_problems: unknown problem {name!r} (s1, s2 or co)")
        bits |= SAMPLE_BITS[name]
    return RpSampleOpts(int(num), int(seed) & (2 ** 64 - 1), bits)


def dot_bracket(table) -> str:
    """Dot-bracket string of a pair table (t[k-1] = 1-based partner of base k, 0 unpaired)."""
    t = np.asarray(table)
    return "".join("." if p == 0 else ("(" if p > k + 1 else ")") for k, p in enumerate(t.tolist()))


def joint_structure(co_table, n1: int) -> Tuple[str, str]:
    """A co-fold sample (pair table over s1 s2, s2's base b at n1 + b) in RactIP's notation for a joint structure:
    () intramolecular, [ in s1 and ] in s2 for a pair that joins the strands (the k-th [ from the 3' end of s1 with the
    k-th ] from the 5' end of s2).  The result is a valid -c constraint line for the pair."""
    t = np.asarray(co_table).tolist()
    out = []
    for k, p in enumerate(t, start=1):
        if p == 0:
            out.append(".")
        elif (k <= n1) != (p <= n1):
            out.append("[" if k <= n1 else "]")
        else:
            out.append("(" if p > k else ")")
    s = "".join(out)
    return s[:n1], s[n1:]


class DeviceBatch:
    """A batch whose inputs are resident in HBM (rp_batch_*).  constraints: None, or one (c1, c2) per pair -- the
    structure constraints of rp_batch_create_constrained, either string (or the whole entry) None for none.
    stack_energies: None, or one (e1, e2) per pair -- stacking pseudo-energies in kcal/mol over s1 and s2
    (rp_batch_create_soft, e.g. from shape_deigan), either array (or the whole entry) None for none.
    samples > 0: every run also draws that many structures of each of sample_problems ("s1", "s2", "co") with
    sample_seed (rp_batch_create_sampled); fetch_samples() and sample_tensors() return them.
    unpaired_energies: None, or one (u1, u2) per pair -- unpaired pseudo-energies in kcal/mol over s1 and s2
    (rp_batch_create_probed, RNAfold --shapeMethod=W), either array (or the whole entry) None for none."""

    def __init__(self, stage: "ProbabilityStage", pairs: Sequence[Tuple[str, str]], opts: RpOpts,
                 constraints: Optional[Sequence[Optional[Tuple[Optional[str], Optional[str]]]]] = None,
                 stack_energies=None, samples: int = 0, sample_seed: int = 1,
                 sample_problems: Sequence[str] = ("s1", "s2", "co"), unpaired_energies=None):
        self.stage, self.lib, self.opts = stage, stage.lib, opts
        self.pairs = list(pairs)
        self.n = len(self.pairs)
        arr, keep = _make_pairs(self.pairs)
        self.layout = (RpDenseLayout * max(self.n, 1))()
        tot = C.c_size_t()
        stage._check(self.lib.rp_dense_plan(arr, self.n, C.byref(opts), self.layout, C.byref(tot)))
        self.total_floats = tot.value
        self.slayout = (RpSparseLayout * max(self.n, 1))()
        tr, tf = C.c_size_t(), C.c_size_t()
        stage._check(self.lib.rp_sparse_plan(arr, self.n, C.byref(opts), self.slayout, C.byref(tr), C.byref(tf)))
        self.total_recs, self.total_upf = tr.value, tf.value
        self.handle = C.c_void_p()
        self.samples = int(samples)
        self.sample_layout = (RpSampleLayout * max(self.n, 1))()
        self.total_samples = 0
        if self.samples != 0 or unpaired_energies is not None:
            so = sample_opts(self.samples, sample_seed, sample_problems)
            cons, ckeep = _make_constraints(constraints, self.n) if constraints is not None else (None, None)
            se, ekeep = (_make_stack_energies(stack_energies, self.pairs) if stack_energies is not None
                         else (None, None))
            if unpaired_energies is None:
                stage._check(self.lib.rp_batch_create_sampled(stage.ctx, arr, cons, se, self.n, C.byref(opts),
                                                              C.byref(so), C.byref(self.handle)))
            else:
                ue, ukeep = _make_energies(unpaired_energies, self.pairs, RpUnpairedEnergy, "unpaired_energies", "u")
                stage._check(self.lib.rp_batch_create_probed(stage.ctx, arr, cons, se, ue, self.n, C.byref(opts),
                                                             C.byref(so), C.byref(self.handle)))
            ts = C.c_size_t()
            stage._check(self.lib.rp_sample_plan(arr, self.n, C.byref(so), self.sample_layout, C.byref(ts)))
            self.total_samples = ts.value
        elif stack_energies is not None:
            cons, ckeep = _make_constraints(constraints, self.n) if constraints is not None else (None, None)
            se, ekeep = _make_stack_energies(stack_energies, self.pairs)
            stage._check(self.lib.rp_batch_create_soft(stage.ctx, arr, cons, se, self.n, C.byref(opts),
                                                       C.byref(self.handle)))
        elif constraints is None:
            stage._check(self.lib.rp_batch_create(stage.ctx, arr, self.n, C.byref(opts), C.byref(self.handle)))
        else:
            cons, ckeep = _make_constraints(constraints, self.n)
            stage._check(self.lib.rp_batch_create_constrained(stage.ctx, arr, cons, self.n, C.byref(opts),
                                                              C.byref(self.handle)))

    def run(self):
        self.stage._check(self.lib.rp_batch_run(self.handle))

    def sync(self):
        self.stage._check(self.lib.rp_batch_sync(self.handle))

    def fetch_dense(self, out: Optional[np.ndarray] = None) -> np.ndarray:
        if out is None:
            out = np.empty(max(self.total_floats, 1), dtype=np.float32)
        self.stage._check(self.lib.rp_batch_fetch_dense(self.handle, out.ctypes.data, out.size))
        return out

    def fetch_sparse(self, recs=None, ups=None, counts=None, with_ups: bool = True):
        """Thresholded lists x, y, z, v, w (+ the dense window tables unless with_ups=False).
        counts[k] = (n_x, n_y, n_z, overflow, n_v, n_w)."""
        if recs is None:
            recs = np.zeros(max(self.total_recs, 1), dtype=REC_DTYPE)
        if ups is None and with_ups:
            ups = np.empty(max(self.total_upf, 1), dtype=np.float32)
        if counts is None:
            counts = np.zeros((max(self.n, 1), 6), dtype=np.int32)
        self.stage._check(self.lib.rp_batch_fetch_sparse(self.handle, recs.ctypes.data, recs.size,
                                                         C.c_void_p(ups.ctypes.data if ups is not None else 0),
                                                         ups.size if ups is not None else 0, counts.ctypes.data))
        return recs, ups, counts

    def fetch_logz(self) -> np.ndarray:
        lz = np.zeros((max(self.n, 1), 3))
        self.stage._check(self.lib.rp_batch_fetch_logz(self.handle, lz.ctypes.data, lz.size))
        return lz[:self.n]

    def fetch_samples(self) -> List[Dict[str, np.ndarray]]:
        """The samples of the last run: per pair, {problem: int16 [num, n]} for each sampled problem ("s1", "s2",
        "co"; n = n1, n2, n1+n2), each row a pair table (t[k-1] = 1-based partner of base k, 0 unpaired)."""
        flat = np.zeros(max(self.total_samples, 1), dtype=np.int16)
        self.stage._check(self.lib.rp_batch_fetch_samples(self.handle, flat.ctypes.data, flat.size))
        out = []
        for k, (s1, s2) in enumerate(self.pairs):
            L = self.sample_layout[k]
            d = {}
            for name, off, ln, n in (("s1", L.s1, L.len_s1, len(s1)), ("s2", L.s2, L.len_s2, len(s2)),
                                     ("co", L.co, L.len_co, len(s1) + len(s2))):
                if ln:
                    d[name] = flat[off:off + ln].reshape(self.samples, n)
            out.append(d)
        return out

    def sample_tensors(self) -> Dict[str, "torch.Tensor"]:
        """The samples as padded int16 CUDA tensors s1 [B, num, N1], s2 [B, num, N2], co [B, num, N1+N2] (N1 / N2 the
        longest first / second sequence of the batch), zero past each pair's own length and for problems that were
        not sampled.  Copied on the device and enqueued on torch's current stream, like dense_tensor()."""
        B, num = self.n, self.samples
        N1 = max([len(a) for a, _ in self.pairs], default=0)
        N2 = max([len(b) for _, b in self.pairs], default=0)
        with self.stage._torch_stream() as torch:
            dev = self.stage.torch_device()
            flat = torch.empty(max(self.total_samples, 1), dtype=torch.int16, device=dev)
            self.stage._check(self.lib.rp_batch_samples_device(self.handle, C.c_void_p(flat.data_ptr()), flat.numel()))
            out = {"s1": torch.zeros((B, num, N1), dtype=torch.int16, device=dev),
                   "s2": torch.zeros((B, num, N2), dtype=torch.int16, device=dev),
                   "co": torch.zeros((B, num, N1 + N2), dtype=torch.int16, device=dev)}
            for k, (s1, s2) in enumerate(self.pairs):
                L = self.sample_layout[k]
                for name, off, ln, n in (("s1", L.s1, L.len_s1, len(s1)), ("s2", L.s2, L.len_s2, len(s2)),
                                         ("co", L.co, L.len_co, len(s1) + len(s2))):
                    if ln:
                        out[name][k, :, :n] = flat[off:off + ln].view(num, n)
        return out

    def square_layout(self) -> RpSquareLayout:
        """rp_square_plan of the batch: B, N1, N2, W and the element count of each square tensor."""
        arr, keep = _make_pairs(self.pairs)
        lay = RpSquareLayout()
        self.stage._check(self.lib.rp_square_plan(arr, self.n, C.byref(self.opts), C.byref(lay)))
        return lay

    def dense_tensor(self):
        """The dense outputs as one flat float32 CUDA tensor in the layout of rp_dense_plan (the values
        fetch_dense() returns), copied on the device.  Enqueued on torch's current stream: torch ops that
        follow on that stream see the result without a host synchronisation."""
        with self.stage._torch_stream() as torch:
            out = torch.empty(max(self.total_floats, 1), dtype=torch.float32, device=self.stage.torch_device())
            self.stage._check(self.lib.rp_batch_dense_device(self.handle, C.c_void_p(out.data_ptr()), out.numel()))
        return out[:self.total_floats]

    def tensors(self) -> Dict[str, "torch.Tensor"]:
        """The outputs as padded square float32 CUDA tensors (rp_batch_square_device), 1-based like the reference:
        bp1 [B, N1+1, N1+1] and bp2 [B, N2+1, N2+1] symmetric, up1 [B, N1, W], up2 [B, N2, W], hp [B, N1+1, N2+1],
        N1 / N2 the longest first / second sequence of the batch, W = max_w; index 0 and everything past a pair's
        own lengths are 0.  n1 and n2 (int32 [B]) hold each pair's lengths for masking.  Enqueued on torch's
        current stream, like dense_tensor()."""
        lay = self.square_layout()
        B, N1, N2, W = lay.B, lay.N1, lay.N2, lay.W
        shapes = {"bp1": (B, N1 + 1, N1 + 1), "bp2": (B, N2 + 1, N2 + 1), "up1": (B, N1, W), "up2": (B, N2, W),
                  "hp": (B, N1 + 1, N2 + 1)}
        with self.stage._torch_stream() as torch:
            dev = self.stage.torch_device()
            out = {k: torch.empty(shapes[k], dtype=torch.float32, device=dev) for k in SQUARE_KEYS}
            ptrs = [C.c_void_p(out[k].data_ptr() if out[k].numel() else None) for k in SQUARE_KEYS]
            self.stage._check(self.lib.rp_batch_square_device(self.handle, *ptrs))
            lens = torch.tensor([len(a) for a, _ in self.pairs] + [len(b) for _, b in self.pairs], dtype=torch.int32)
            lens = lens.pin_memory().to(dev, non_blocking=True)
        out["n1"], out["n2"] = lens[:self.n], lens[self.n:]
        return out

    def split_dense(self, flat: np.ndarray) -> List[PairProbabilities]:
        out = []
        w = max(self.opts.max_w, 0)
        for k, (s1, s2) in enumerate(self.pairs):
            L = self.layout[k]
            n1, n2 = len(s1), len(s2)
            out.append(PairProbabilities(
                bp1=flat[L.bp1:L.bp1 + L.n_bp1], offset1=bp_offsets(n1),
                up1=flat[L.up1:L.up1 + L.n_up1].reshape(n1, w),
                bp2=flat[L.bp2:L.bp2 + L.n_bp2], offset2=bp_offsets(n2),
                up2=flat[L.up2:L.up2 + L.n_up2].reshape(n2, w),
                hp=flat[L.hp:L.hp + L.n_hp].reshape(n1 + 1, n2 + 1)))
        return out

    def split_sparse(self, recs, ups, counts) -> List[PairRecords]:
        out = []
        w = max(self.opts.max_w, 0)
        for k, (s1, s2) in enumerate(self.pairs):
            S = self.slayout[k]
            nx, ny, nz, nv, nw = (int(counts[k][0]), int(counts[k][1]), int(counts[k][2]), int(counts[k][4]),
                                  int(counts[k][5]))
            out.append(PairRecords(
                x=recs[S.x:S.x + nx], y=recs[S.y:S.y + ny], z=recs[S.z:S.z + nz],
                up1=None if ups is None else ups[S.up1:S.up1 + S.n_up1].reshape(len(s1), w),
                up2=None if ups is None else ups[S.up2:S.up2 + S.n_up2].reshape(len(s2), w),
                v=recs[S.v:S.v + nv], w=recs[S.w:S.w + nw]))
        return out

    def close(self):
        if self.handle:
            self.lib.rp_batch_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ProbabilityStage:
    """One context per process per GPU.  Raises if the CUDA library or a GPU is
    missing -- the stage has no CPU fallback."""

    def __init__(self, model: Optional[RpModel] = None, device: int = 0, use_bl: bool = True,
                 param_file: Optional[str] = None):
        self.lib = _lib.load()
        self.model = model if model is not None else default_model(use_bl, param_file)
        self.ctx = C.c_void_p()
        rc = self.lib.rp_create(C.byref(self.ctx), C.byref(self.model), device)
        if rc:
            raise RpError(rc, self.lib.rp_last_error(None).decode() or self.lib.rp_strerror(rc).decode())
        self.device = device

    def _check(self, rc: int):
        if rc:
            msg = self.lib.rp_last_error(self.ctx).decode() or self.lib.rp_strerror(rc).decode()
            raise RpError(rc, msg)

    def torch_device(self):
        import torch
        return torch.device("cuda", self.device)

    @contextlib.contextmanager
    def _torch_stream(self):
        """Run the block's library calls on torch's current stream, then give the context its previous stream
        back.  torch is imported here only: the rest of the stage works without it."""
        import torch
        if torch.cuda.current_device() != self.device:
            raise RuntimeError(f"torch's current device is cuda:{torch.cuda.current_device()}, this stage runs on "
                               f"cuda:{self.device}: select it with torch.cuda.device({self.device})")
        prev = C.c_void_p()
        self._check(self.lib.rp_get_stream(self.ctx, C.byref(prev)))
        stream = torch.cuda.current_stream(self.device).cuda_stream or _CUDA_STREAM_LEGACY
        self._check(self.lib.rp_set_stream(self.ctx, C.c_void_p(stream)))
        try:
            yield torch
        finally:
            self.lib.rp_set_stream(self.ctx, prev)

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.rp_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------- minimum free energy
    def mfe(self, pairs: Sequence[Tuple[str, str]], constraints=None, stack_energies=None, unpaired_energies=None,
            problems: Sequence[str] = ("s1", "s2", "co")) -> List[Dict[str, Tuple[np.ndarray, float]]]:
        """rp_run_mfe: per pair {problem: (int16 pair table, MFE in kcal/mol)} for each of `problems` ("s1", "s2",
        "co"; a pair with an empty s2 has s1 only).  constraints, stack_energies, unpaired_energies as DeviceBatch
        takes them.  The co-fold's table runs over s1 s2 (joint_structure turns it into RactIP's notation) and its
        energy counts DuplexInit when a pair joins the strands, as energy_of_duplex does."""
        pairs = list(pairs)
        n = len(pairs)
        so = sample_opts(1, 1, problems)
        arr, keep = _make_pairs(pairs)
        cons, ckeep = _make_constraints(constraints, n) if constraints is not None else (None, None)
        se, ekeep = _make_stack_energies(stack_energies, pairs) if stack_energies is not None else (None, None)
        ue, ukeep = (_make_energies(unpaired_energies, pairs, RpUnpairedEnergy, "unpaired_energies", "u")
                     if unpaired_energies is not None else (None, None))
        layout = (RpSampleLayout * max(n, 1))()
        tot = C.c_size_t()
        self._check(self.lib.rp_sample_plan(arr, n, C.byref(so), layout, C.byref(tot)))
        tables = np.zeros(max(tot.value, 1), dtype=np.int16)
        energies = np.zeros(max(3 * n, 1), dtype=np.int32)
        self._check(self.lib.rp_run_mfe(self.ctx, arr, cons, se, ue, n, so.problems, tables.ctypes.data, tot.value,
                                        energies.ctypes.data))
        out = []
        for k in range(n):
            L = layout[k]
            d = {}
            for w, (name, off, ln) in enumerate((("s1", L.s1, L.len_s1), ("s2", L.s2, L.len_s2), ("co", L.co, L.len_co))):
                if ln:
                    d[name] = (tables[off:off + ln].copy(), int(energies[3 * k + w]) / 100.0)
            out.append(d)
        return out

    # ------------------------------------------------------------- batches
    def batch(self, pairs: Sequence[Tuple[str, str]], opts: Optional[RpOpts] = None,
              constraints=None, stack_energies=None, samples: int = 0, sample_seed: int = 1,
              sample_problems: Sequence[str] = ("s1", "s2", "co"), unpaired_energies=None) -> DeviceBatch:
        """constraints: None, or one (c1, c2) structure-constraint pair per pair; stack_energies: None, or one (e1, e2)
        pair of stacking pseudo-energy arrays per pair; samples, sample_seed, sample_problems: stochastic samples;
        unpaired_energies: None, or one (u1, u2) pair of unpaired pseudo-energy arrays per pair (DeviceBatch)."""
        return DeviceBatch(self, pairs, opts if opts is not None else default_opts(), constraints, stack_energies,
                           samples, sample_seed, sample_problems, unpaired_energies)

    def run_dense(self, pairs: Sequence[Tuple[str, str]], opts: Optional[RpOpts] = None,
                  pinned: bool = False, constraints=None, stack_energies=None,
                  unpaired_energies=None) -> List[PairProbabilities]:
        """rp_run_dense: host buffers in, host buffers out.  pinned=True hands the library a page-locked
        buffer (rp_host_alloc) as the target of its device-to-host copy.  With constraints, stack_energies or
        unpaired_energies (one entry per pair, see DeviceBatch) the pairs run as a device batch that carries them."""
        opts = opts if opts is not None else default_opts()
        if constraints is not None or stack_energies is not None or unpaired_energies is not None:
            b = self.batch(pairs, opts, constraints, stack_energies, unpaired_energies=unpaired_energies)
            try:
                b.run()
                return b.split_dense(b.fetch_dense())
            finally:
                b.close()
        arr, keep = _make_pairs(pairs)
        n = len(pairs)
        layout = (RpDenseLayout * max(n, 1))()
        tot = C.c_size_t()
        self._check(self.lib.rp_dense_plan(arr, n, C.byref(opts), layout, C.byref(tot)))
        if pinned:
            nfl = max(tot.value, 1)
            ptr = self.lib.rp_host_alloc(nfl * 4)
            if not ptr:
                raise MemoryError("rp_host_alloc failed")
            try:
                self._check(self.lib.rp_run_dense(self.ctx, arr, n, C.byref(opts), C.c_void_p(ptr), nfl))
                flat = np.ctypeslib.as_array((C.c_float * nfl).from_address(ptr)).copy()
            finally:
                self.lib.rp_host_free(C.c_void_p(ptr))
        else:
            flat = np.empty(max(tot.value, 1), dtype=np.float32)
            self._check(self.lib.rp_run_dense(self.ctx, arr, n, C.byref(opts), flat.ctypes.data, flat.size))
        w = max(opts.max_w, 0)
        out = []
        for k, (s1, s2) in enumerate(pairs):
            L = layout[k]
            n1, n2 = len(s1), len(s2)
            out.append(PairProbabilities(
                bp1=flat[L.bp1:L.bp1 + L.n_bp1], offset1=bp_offsets(n1),
                up1=flat[L.up1:L.up1 + L.n_up1].reshape(n1, w),
                bp2=flat[L.bp2:L.bp2 + L.n_bp2], offset2=bp_offsets(n2),
                up2=flat[L.up2:L.up2 + L.n_up2].reshape(n2, w),
                hp=flat[L.hp:L.hp + L.n_hp].reshape(n1 + 1, n2 + 1)))
        return out

    def run_tensors(self, pairs: Sequence[Tuple[str, str]], opts: Optional[RpOpts] = None) -> Dict[str, "torch.Tensor"]:
        """batch + run + DeviceBatch.tensors(): the square CUDA tensors of `pairs`.  Closing the batch waits for
        the expansion (the batch's buffers go back to the context's pool)."""
        b = self.batch(pairs, opts)
        try:
            b.run()
            return b.tensors()
        finally:
            b.close()

    def run_sparse(self, pairs: Sequence[Tuple[str, str]], opts: Optional[RpOpts] = None,
                   constraints=None, stack_energies=None, unpaired_energies=None) -> List[PairRecords]:
        opts = opts if opts is not None else default_opts()
        b = self.batch(pairs, opts, constraints, stack_energies, unpaired_energies=unpaired_energies)
        try:
            b.run()
            return b.split_sparse(*b.fetch_sparse())
        finally:
            b.close()

    # --------------------------------------- the reference's three calls
    def solve_probabilities(self, s1: str, s2: str, opts: Optional[RpOpts] = None) -> PairProbabilities:
        """rnafold(fa1), rnafold(fa2), rnaduplex(fa1, fa2)  (src/ractip.cpp:546-548)."""
        return self.run_dense([(s1, s2)], opts)[0]

    def rnafold(self, seq: str, max_w: int = 15):
        """RactIP::rnafold (src/ractip.cpp:308-382): (bp, offset, up).  A pair with an empty second
        sequence computes s1's sections only."""
        r = self.run_dense([(seq, "")], default_opts(max_w=max(1, max_w)))[0]
        return r.bp1, r.offset1, r.up1

    def rnaduplex(self, s1: str, s2: str, th_hy: float = 0.1, use_pf_duplex: bool = False) -> np.ndarray:
        """RactIP::rnaduplex (src/ractip.cpp:384-459): hp."""
        return self.run_dense([(s1, s2)], default_opts(th_hy=th_hy, use_pf_duplex=int(use_pf_duplex)))[0].hp

    # ------------------------------------------------------------ utilities
    def last_timing(self) -> RpTiming:
        t = RpTiming()
        self._check(self.lib.rp_last_timing(self.ctx, C.byref(t)))
        return t

    def measure_peaks(self) -> Tuple[float, float]:
        f, s = C.c_double(), C.c_double()
        self._check(self.lib.rp_measure_peaks(self.ctx, C.byref(f), C.byref(s)))
        return f.value, s.value


def zscore_shuffles(s1: str, s2: str, num: int, seed: int, mode: int = 12, k: int = 2):
    """The shuffled sequences of the --zscore loop (src/ractip.cpp:1636-1643)."""
    lib = _lib.load()
    b1, b2 = s1.encode(), s2.encode()
    o1 = C.create_string_buffer(max(1, num * len(b1)))
    o2 = C.create_string_buffer(max(1, num * len(b2)))
    rc = lib.rp_zscore_shuffles(b1, len(b1), b2, len(b2), mode, seed, num, k, o1, o2)
    if rc:
        raise RpError(rc, lib.rp_strerror(rc).decode())
    r1 = [o1.raw[r * len(b1):(r + 1) * len(b1)].decode() for r in range(num)]
    r2 = [o2.raw[r * len(b2):(r + 1) * len(b2)].decode() for r in range(num)]
    return r1, r2
