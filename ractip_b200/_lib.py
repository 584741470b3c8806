"""ctypes binding of libractip_prob.so (the C ABI in include/ractip_prob.h).

The library is built in-tree by ractip_b200/build.py.  Loading fails loudly if
it is missing: there is no Python or CPU fallback for the probability stage.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libractip_prob.so"

NB = 7


class RpModel(C.Structure):
    _fields_ = [
        ("temperature", C.c_double),
        ("dangles", C.c_int),
        ("special_hp", C.c_int),
        ("pf_smooth", C.c_int),
        ("sfact", C.c_double),
        ("stack37", (C.c_int * 8) * 8),
        ("hairpin37", C.c_int * 31),
        ("bulge37", C.c_int * 31),
        ("internal_loop37", C.c_int * 31),
        ("mismatchI37", ((C.c_int * 5) * 5) * 8),
        ("mismatchH37", ((C.c_int * 5) * 5) * 8),
        ("mismatchM37", ((C.c_int * 5) * 5) * 8),
        ("mismatchExt37", ((C.c_int * 5) * 5) * 8),
        ("mismatch1nI37", ((C.c_int * 5) * 5) * 8),
        ("mismatch23I37", ((C.c_int * 5) * 5) * 8),
        ("dangle5_37", (C.c_int * 5) * 8),
        ("dangle3_37", (C.c_int * 5) * 8),
        ("int11_37", (((C.c_int * 5) * 5) * 8) * 8),
        ("int21_37", ((((C.c_int * 5) * 5) * 5) * 8) * 8),
        ("int22_37", (((((C.c_int * 5) * 5) * 5) * 5) * 8) * 8),
        ("ML_BASE37", C.c_int),
        ("ML_closing37", C.c_int),
        ("ML_intern37", C.c_int),
        ("TerminalAU37", C.c_int),
        ("ninio37", C.c_int),
        ("MAX_NINIO", C.c_int),
        ("DuplexInit37", C.c_int),
        ("lxc37", C.c_double),
        ("Tetraloops", C.c_char * 1401),
        ("Tetraloop37", C.c_int * 200),
        ("Triloops", C.c_char * 241),
        ("Triloop37", C.c_int * 40),
        ("Hexaloops", C.c_char * 1801),
        ("Hexaloop37", C.c_int * 200),
    ]


class RpPair(C.Structure):
    _fields_ = [("s1", C.c_char_p), ("n1", C.c_int), ("s2", C.c_char_p), ("n2", C.c_int)]


class RpConstraint(C.Structure):
    _fields_ = [("c1", C.c_char_p), ("c2", C.c_char_p)]


class RpOpts(C.Structure):
    _fields_ = [("max_w", C.c_int), ("min_w", C.c_int), ("th_ss", C.c_float), ("th_hy", C.c_float),
                ("th_ac", C.c_float), ("use_pf_duplex", C.c_int)]


class RpDenseLayout(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in
                ("bp1", "bp2", "up1", "up2", "hp", "n_bp1", "n_bp2", "n_up1", "n_up2", "n_hp")]


class RpSquareLayout(C.Structure):
    _fields_ = [("B", C.c_int), ("N1", C.c_int), ("N2", C.c_int), ("W", C.c_int)] + \
        [(n, C.c_size_t) for n in ("n_bp1", "n_bp2", "n_up1", "n_up2", "n_hp")]


class RpRec(C.Structure):
    _fields_ = [("i", C.c_int32), ("j", C.c_int32), ("p", C.c_float)]


class RpSparseLayout(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in
                ("x", "y", "z", "cap_x", "cap_y", "cap_z", "up1", "up2", "n_up1", "n_up2", "v", "w", "cap_v", "cap_w")]


class RpSparseCounts(C.Structure):
    _fields_ = [("n_x", C.c_int32), ("n_y", C.c_int32), ("n_z", C.c_int32), ("overflow", C.c_int32),
                ("n_v", C.c_int32), ("n_w", C.c_int32)]


class RpIpOpts(C.Structure):
    """rp_ip_opts (include/ractip_ip.h): the RactIP members that shape the integer programme."""
    _fields_ = [("alpha", C.c_float), ("beta", C.c_float), ("th_ss", C.c_float), ("th_hy", C.c_float),
                ("th_ac", C.c_float), ("max_w", C.c_int), ("min_w", C.c_int), ("acc_max", C.c_int),
                ("acc_max_ss", C.c_int), ("acc_num", C.c_int), ("in_pk", C.c_int), ("stacking", C.c_int)]


class RpTiming(C.Structure):
    _fields_ = [("ms_total", C.c_float), ("ms_h2d", C.c_float), ("ms_d2h", C.c_float),
                ("kernel_launches", C.c_int), ("alg_flops", C.c_double),
                ("dominant_kind", C.c_int), ("ms_dominant", C.c_float), ("alg_flops_dominant", C.c_double)]


# every symbol include/ractip_prob.h declares (tests check the .so exports all)
EXPORTS = [
    "rp_model_default", "rp_model_read_par", "rp_model_digest", "rp_opts_default",
    "rp_dense_plan", "rp_sparse_plan", "rp_create", "rp_destroy", "rp_last_error",
    "rp_strerror", "rp_set_stream", "rp_get_stream", "rp_host_alloc", "rp_host_free", "rp_run_dense",
    "rp_run_sparse", "rp_batch_create", "rp_batch_create_constrained", "rp_batch_run", "rp_batch_sync",
    "rp_batch_fetch_dense", "rp_batch_fetch_sparse", "rp_batch_sparse_device", "rp_batch_dense_device",
    "rp_square_plan", "rp_batch_square_device", "rp_batch_fetch_logz",
    "rp_batch_destroy", "rp_last_timing", "rp_measure_peaks", "rp_zscore_shuffles",
    "rp_alg_flops_mcc", "rp_version", "rp_kernel_plan",
    "rp_multi_create", "rp_multi_destroy", "rp_multi_devices", "rp_multi_last_error", "rp_multi_run_dense",
    "rp_multi_run_sparse",
    # include/ractip_ip.h (host-side consumer: integer programme, energy evaluation)
    "rp_ip_opts_default", "rp_ip_build", "rp_ip_build_sparse", "rp_ip_build_ss", "rp_ip_dims", "rp_ip_export",
    "rp_ip_decode", "rp_ip_free", "rp_energy_of_structure", "rp_energy_of_duplex",
    # include/ractip_io.h (many-pair front end: the reference's FASTA reader)
    "rp_fasta_load", "rp_fasta_parse", "rp_fasta_count", "rp_fasta_get", "rp_fasta_free",
]

_lib = None


def load() -> C.CDLL:
    """Load the shared library, or raise: the product has no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    import os
    path = Path(os.environ.get("RP_LIB", LIB_PATH))   # RP_LIB: e.g. the tuning build (RP_BUILD_TUNE=1, profile probes compiled in)
    if not path.exists():
        raise ImportError(
            f"{path} is missing: build it with `python -m ractip_b200.build` "
            "(there is no CPU/Python fallback for the probability stage)")
    lib = C.CDLL(str(path))
    vp, i, sz = C.c_void_p, C.c_int, C.c_size_t
    P = C.POINTER
    sig = {
        "rp_model_default": (i, [P(RpModel), i]),
        "rp_model_read_par": (i, [P(RpModel), C.c_char_p]),
        "rp_model_digest": (C.c_uint64, [P(RpModel)]),
        "rp_opts_default": (None, [P(RpOpts)]),
        "rp_dense_plan": (i, [P(RpPair), i, P(RpOpts), P(RpDenseLayout), P(sz)]),
        "rp_sparse_plan": (i, [P(RpPair), i, P(RpOpts), P(RpSparseLayout), P(sz), P(sz)]),
        "rp_create": (i, [P(vp), P(RpModel), i]),
        "rp_destroy": (i, [vp]),
        "rp_last_error": (C.c_char_p, [vp]),
        "rp_strerror": (C.c_char_p, [i]),
        "rp_set_stream": (i, [vp, vp]),
        "rp_get_stream": (i, [vp, P(vp)]),
        "rp_host_alloc": (vp, [sz]),
        "rp_host_free": (None, [vp]),
        "rp_run_dense": (i, [vp, P(RpPair), i, P(RpOpts), vp, sz]),
        "rp_run_sparse": (i, [vp, P(RpPair), i, P(RpOpts), vp, sz, vp, sz, vp]),
        "rp_batch_create": (i, [vp, P(RpPair), i, P(RpOpts), P(vp)]),
        "rp_batch_create_constrained": (i, [vp, P(RpPair), P(RpConstraint), i, P(RpOpts), P(vp)]),
        "rp_batch_run": (i, [vp]),
        "rp_batch_sync": (i, [vp]),
        "rp_batch_fetch_dense": (i, [vp, vp, sz]),
        "rp_batch_fetch_sparse": (i, [vp, vp, sz, vp, sz, vp]),
        "rp_batch_sparse_device": (i, [vp, vp, sz, vp, sz, vp]),
        "rp_batch_dense_device": (i, [vp, vp, sz]),
        "rp_square_plan": (i, [P(RpPair), i, P(RpOpts), P(RpSquareLayout)]),
        "rp_batch_square_device": (i, [vp, vp, vp, vp, vp, vp]),
        "rp_batch_fetch_logz": (i, [vp, vp, sz]),
        "rp_batch_destroy": (i, [vp]),
        "rp_last_timing": (i, [vp, P(RpTiming)]),
        "rp_measure_peaks": (i, [vp, P(C.c_double), P(C.c_double)]),
        "rp_zscore_shuffles": (i, [C.c_char_p, i, C.c_char_p, i, i, C.c_uint, i, i, C.c_char_p, C.c_char_p]),
        "rp_alg_flops_mcc": (C.c_double, [i]),
        "rp_version": (C.c_char_p, []),
        "rp_kernel_plan": (i, [i, sz, P(sz)]),
        "rp_multi_create": (i, [P(vp), P(RpModel), P(i), i]),
        "rp_multi_destroy": (i, [vp]),
        "rp_multi_devices": (i, [vp]),
        "rp_multi_last_error": (C.c_char_p, [vp]),
        "rp_multi_run_dense": (i, [vp, P(RpPair), i, P(RpOpts), vp, sz]),
        "rp_multi_run_sparse": (i, [vp, P(RpPair), i, P(RpOpts), vp, sz, vp]),
        "rp_ip_opts_default": (None, [P(RpIpOpts)]),
        "rp_ip_build": (i, [P(RpIpOpts), i, i, vp, vp, vp, vp, vp, P(vp)]),
        "rp_ip_build_sparse": (i, [P(RpIpOpts), i, i, vp, i, vp, i, vp, i, vp, i, vp, i, P(vp)]),
        "rp_ip_build_ss": (i, [P(RpIpOpts), i, vp, vp, P(vp)]),
        "rp_ip_dims": (i, [vp, P(i), P(i), P(i)]),
        "rp_ip_export": (i, [vp, vp, vp, vp, vp, vp, vp, vp]),
        "rp_ip_decode": (i, [vp, vp, C.c_char_p, C.c_char_p, vp, vp]),
        "rp_ip_free": (None, [vp]),
        "rp_energy_of_structure": (i, [P(RpModel), C.c_char_p, C.c_char_p, i, i, P(C.c_float)]),
        "rp_energy_of_duplex": (i, [P(RpModel), C.c_char_p, i, C.c_char_p, i, C.c_char_p, C.c_char_p, P(C.c_float)]),
        "rp_fasta_load": (i, [C.c_char_p, P(vp)]),
        "rp_fasta_parse": (i, [C.c_char_p, sz, P(vp)]),
        "rp_fasta_count": (i, [vp]),
        "rp_fasta_get": (i, [vp, i, P(C.c_char_p), P(C.c_char_p), P(C.c_char_p)]),
        "rp_fasta_free": (None, [vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
