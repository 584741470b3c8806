"""Energy-model layer: BL* copy semantics (reference src/boltzmann_param.c:5908-6026),
the embedded Turner-2004 residual tables and the -P reader."""
import ctypes as C
import struct
from pathlib import Path

import numpy as np

# The reference's BL* initialisers (src/boltzmann_param.c:21-5906, macros expanded), frozen: a byte copy of
# params/blstar.bin as tools/gen_blstar_bin.py wrote it from that source, which this test had checked it against.
# Kept apart from params/ so that an edit of the product's tables cannot move the expectation with it.
BLSTAR_REF = Path(__file__).resolve().parent / "golden" / "blstar_reference.bin"
INF = 10000000


def test_default_model_values(lib, model):
    m = model
    # BL* scalars: src/boltzmann_param.c:5857-5868
    assert (m.ML_BASE37, m.ML_closing37, m.ML_intern37, m.TerminalAU37) == (-2, 315, 15, 56)
    assert (m.ninio37, m.MAX_NINIO) == (50, 300)
    # stack37a first row: src/boltzmann_param.c:23
    assert [m.stack37[1][j] for j in range(1, 8)] == [-133, -207, -146, -37, -139, -132, 0]
    # copy_dangle fills row 0 and column 0 with INF (src/boltzmann_param.c:113-120,5965-5971)
    assert m.dangle5_37[0][0] == INF and m.dangle5_37[1][0] == INF and m.dangle5_37[1][1] == -8
    assert m.dangle3_37[7][0] == 0
    # tetraloop list replaced by the 30 BL* entries (src/boltzmann_param.c:5875-5904,5995-6008)
    tl = m.Tetraloops.decode()
    assert len(tl) == 210 and tl.startswith("GGGGAC GGUGAC ") and tl.endswith("UGGAAA ")
    assert m.Tetraloop37[0] == -33 and m.Tetraloop37[29] == 1 and m.Tetraloop37[30] == 0
    # untouched Turner-2004 residuals
    assert m.DuplexInit37 == 410 and abs(m.lxc37 - 107.856) < 1e-12
    assert m.Triloops.decode() == "CAACG GUUAC " and m.Hexaloops.decode().startswith("ACAGUACU ")
    assert m.temperature == 37.0 and m.dangles == 2


def test_default_model_digest_is_stable(lib, model):
    # pins every embedded table: a change in params/ or in the copy logic must be deliberate
    d1 = lib.rp_model_digest(C.byref(model))
    from ractip_b200 import default_model
    d2 = lib.rp_model_digest(C.byref(default_model()))
    assert d1 == d2 and d1 != 0
    golden = Path(__file__).parent / "golden" / "model_digest.txt"
    assert golden.exists(), "run tools/gen_model_digest.py"
    assert int(golden.read_text().strip()) == d1


def _blstar_arrays():
    """name -> values of the frozen reference arrays (the packed layout of tools/gen_blstar_bin.py)."""
    blob = BLSTAR_REF.read_bytes()
    assert blob[:8] == b"RPBLSTR1"
    (n,), p = struct.unpack_from("<i", blob, 8), 12
    arrays = {}
    for _ in range(n):
        name = blob[p:p + 24].rstrip(b"\0").decode()
        (cnt,) = struct.unpack_from("<i", blob, p + 24)
        arrays[name] = list(struct.unpack_from("<%di" % cnt, blob, p + 28))
        p += 28 + 4 * cnt
    return arrays


def test_blstar_matches_reference_source(model):
    """Every BL* array against the reference's own initialisers, with the reference's index ranges."""
    arrays = _blstar_arrays()
    assert {k: len(v) for k, v in arrays.items()} == {
        "stack37a": 49, "mismatchH37a": 175, "mismatchI37a": 175, "dangle5_37a": 40, "dangle3_37a": 40,
        "int11_37a": 1225, "int21_37a": 6125, "int22_37a": 12544, "hairpin37a": 31, "bulge37a": 31,
        "internal_loop37a": 31, "MLparams_a": 4, "ninio_a": 2}
    m = model
    a = arrays["stack37a"]; p = 0
    for i in range(1, 8):
        for j in range(1, 8):
            assert m.stack37[i][j] == a[p]; p += 1
    for name, fld in [("mismatchH37a", m.mismatchH37), ("mismatchI37a", m.mismatchI37)]:
        a = arrays[name]; p = 0
        for i in range(1, 8):
            for j in range(5):
                for k in range(5):
                    assert fld[i][j][k] == a[p]; p += 1
    for name, fld in [("dangle5_37a", m.dangle5_37), ("dangle3_37a", m.dangle3_37)]:
        a = arrays[name]; p = 0
        for i in range(8):
            for j in range(5):
                assert fld[i][j] == a[p]; p += 1
    a = np.array(arrays["int11_37a"]).reshape(7, 7, 5, 5)
    assert np.array_equal(np.ctypeslib.as_array(m.int11_37)[1:, 1:], a)
    a = np.array(arrays["int21_37a"]).reshape(7, 7, 5, 5, 5)
    assert np.array_equal(np.ctypeslib.as_array(m.int21_37)[1:, 1:], a)
    a = np.array(arrays["int22_37a"]).reshape(7, 7, 4, 4, 4, 4)
    assert np.array_equal(np.ctypeslib.as_array(m.int22_37)[1:, 1:, 1:, 1:, 1:, 1:], a)
    for name, fld in [("hairpin37a", m.hairpin37), ("bulge37a", m.bulge37), ("internal_loop37a", m.internal_loop37)]:
        assert list(fld) == arrays[name]


def test_residual_tables_are_self_consistent(model):
    """rna_turner2004.par convention: the N row/column of every mismatch block is the max over ACGU."""
    for fld in (model.mismatchM37, model.mismatchExt37, model.mismatch23I37, model.mismatch1nI37):
        a = np.ctypeslib.as_array(fld)
        for t in range(1, 7):
            blk = a[t]
            assert np.array_equal(blk[0, 1:], blk[1:, 1:].max(axis=0))
            assert np.array_equal(blk[1:, 0], blk[1:, 1:].max(axis=1))
            assert blk[0, 0] == blk[1:, 1:].max()


def test_par_reader_overlays_sections(lib, tmp_path):
    from ractip_b200 import default_model
    m = default_model()
    par = tmp_path / "x.par"
    par.write_text("""## RNAfold parameter file v2.0

# stack
/*  CG     GC     GU     UG     AU     UA     NS  */
  -240   -330   -210   -140   -210   -210   -140    /* CG */
  -330   -340   -250   -150   -220   -240   -150
  -210   -250    130    -50   -140   -130    130
  -140   -150    -50     30    -60   -100     30
  -210   -220   -140    -60   -110    -90    -60
  -210   -240   -130   -100    -90   -130    -90
  -140   -150    130     30    -60    -90    130

# hairpin
   INF   INF   INF   540   560   570   540   600   550   640
   650   660   670   680   690   690   700   710   710   720
   720   730   730   740   740   750   750   750   760   760
   770

# NINIO
/* Ninio = MIN(max, m*|n1-n2| */
/*       m  m_dH     max  */
        60   320     300

# ML_params
/* F = cu*n_unpaired + cc + ci*loop_degree (+TermAU) */
/*      cu      cu_dH       cc      cc_dH       ci      ci_dH  */
         0         0       930      3000       -90      -220

# Misc
/* all parameters are pretty much undocumented */
   410   360    50   370   107.856 0

# Tetraloops
CAACGG     550     690
CCAAGG     330   -1030

#END
""")
    rc = lib.rp_model_read_par(C.byref(m), str(par).encode())
    assert rc == 0
    assert m.stack37[1][1] == -240 and m.stack37[7][7] == 130 and m.stack37[2][1] == -330
    assert m.hairpin37[0] == INF and m.hairpin37[3] == 540 and m.hairpin37[30] == 770
    assert (m.ninio37, m.MAX_NINIO) == (60, 300)
    assert (m.ML_BASE37, m.ML_closing37, m.ML_intern37) == (0, 930, -90)
    assert m.TerminalAU37 == 50
    assert m.Tetraloops.decode() == "CAACGG CCAAGG " and m.Tetraloop37[1] == 330
    # sections that are absent keep their values (BL* int11 etc.)
    assert m.bulge37[1] == default_model().bulge37[1]
    assert lib.rp_model_read_par(C.byref(m), b"/nonexistent.par") == 4  # RP_ERR_IO
    bad = tmp_path / "bad.par"
    bad.write_text("# stack\n1 2 3\n")
    assert lib.rp_model_read_par(C.byref(m), str(bad).encode()) == 5  # RP_ERR_FORMAT


def test_no_bl_needs_a_parameter_file(lib):
    from ractip_b200._lib import RpModel
    m = RpModel()
    assert lib.rp_model_default(C.byref(m), 0) == 6  # RP_ERR_NO_DEFAULTS: fail loudly, never guess
