"""Many-pair front end (SURVEY.md section 8, row f4): FASTA in, joint structures out.

What `ractip` does for ONE pair per process (RactIP::run, src/ractip.cpp:1562-1682) -- read the
sequences, fill the probability matrices, build and solve the integer programme, print names,
sequences and bracket strings, optionally the energies and the z-score -- for any number of pairs
with ONE batch on the GPU for all their probability matrices (and one more for all shuffles of a
z-score run).  The IP itself stays on the host, as in the reference.

    python -m ractip_b200 [options] a.fa b.fa        # first record of each file, as the reference
    python -m ractip_b200 [options] ab.fa            # first two records of one file
    python -m ractip_b200 --all-pairs a.fa b.fa      # every record of a.fa against every record of b.fa
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

from . import _lib
from ._lib import RpIpOpts, RpModel, RpOpts
from .ip import JointPrediction, default_ip_opts, solve_joint, solve_ss, zscore_statistic
from .stage import ProbabilityStage, RpError, default_opts, zscore_shuffles


@dataclass
class FastaRecord:
    name: str
    seq: str
    str: str = ""


def _records(lib, handle) -> List[FastaRecord]:
    out = []
    name, seq, st = C.c_char_p(), C.c_char_p(), C.c_char_p()
    for k in range(lib.rp_fasta_count(handle)):
        lib.rp_fasta_get(handle, k, C.byref(name), C.byref(seq), C.byref(st))
        out.append(FastaRecord(name.value.decode("latin-1"), seq.value.decode("latin-1"), st.value.decode("latin-1")))
    lib.rp_fasta_free(handle)
    return out


def load_fasta(path: str) -> List[FastaRecord]:
    """Fasta::load (src/fa.cpp:37-83) through rp_fasta_load."""
    lib = _lib.load()
    h = C.c_void_p()
    rc = lib.rp_fasta_load(str(path).encode(), C.byref(h))
    if rc:
        raise RpError(rc, f"{path}: cannot be opened")
    return _records(lib, h)


def parse_fasta(text: str) -> List[FastaRecord]:
    lib = _lib.load()
    h = C.c_void_p()
    raw = text.encode("latin-1")
    rc = lib.rp_fasta_parse(raw, len(raw), C.byref(h))
    if rc:
        raise RpError(rc, "rp_fasta_parse")
    return _records(lib, h)


def input_pairs(fa1: str, fa2: Optional[str] = None, all_pairs: bool = False) -> List[Tuple[FastaRecord, FastaRecord]]:
    """The pair(s) a run works on.  Reference rules (src/ractip.cpp:1571-1590): two files -> their first records,
    one file -> its first two; a file without (enough) records is a format error.  all_pairs: the cross product of
    the two files' records (one file: every unordered pair of its records)."""
    l1 = load_fasta(fa1)
    if fa2:
        l2 = load_fasta(fa2)
        if not l1:
            raise ValueError(f"{fa1}: Format error")
        if not l2:
            raise ValueError(f"{fa2}: Format error")
        return [(a, b) for a in l1 for b in l2] if all_pairs else [(l1[0], l2[0])]
    if len(l1) < 2:
        raise ValueError(f"{fa1}: Format error")
    if all_pairs:
        return [(l1[i], l1[j]) for i in range(len(l1)) for j in range(i + 1, len(l1))]
    return [(l1[0], l1[1])]


def constraint_line(rec: FastaRecord) -> Optional[str]:
    """The structure constraint `-c` takes from a record's structure line: None for a record without one, '?' and
    ' ' as '.' (no constraint).  The reader also keeps 'l' and 'e', which have no meaning here: a ValueError, as is a
    line whose length differs from the sequence's.  The rest of the alphabet (.x()[]) goes to the library, which
    checks the brackets (rp_batch_create_constrained)."""
    if not rec.str:
        return None
    for k, ch in enumerate(rec.str):
        if ch in "le":
            raise ValueError(f"{rec.name}: structure constraint '{ch}' at position {k + 1} is not supported")
    if len(rec.str) != len(rec.seq):
        raise ValueError(f"{rec.name}: the structure line has {len(rec.str)} characters, the sequence {len(rec.seq)}")
    return rec.str.replace("?", ".").replace(" ", ".")


@dataclass
class PairResult:
    a: FastaRecord
    b: FastaRecord
    joint: JointPrediction
    e1s: Optional[float] = None   # solve_ss energies (for -e and the z-score)
    e2s: Optional[float] = None
    zscore: Optional[Tuple[float, float]] = None


def _f(x: float) -> str:
    """A float the way the reference's iostream prints it (6 significant digits)."""
    return format(float(x), ".6g")


def format_result(r: PairResult, show_energy: bool = False) -> str:
    """The text RactIP::run prints for a pair (src/ractip.cpp:1604-1621,1665-1668)."""
    j = r.joint
    out = [f">{r.a.name}", r.a.seq, j.r1, f">{r.b.name}", r.b.seq, j.r2]
    if show_energy and j.e1 is not None:
        sg = lambda v: ("+" if v >= 0.0 else "") + _f(v)
        out.append(f"(E: JS= {_f(j.e1 + j.e2 + j.e3)} = {_f(j.e1)}{sg(j.e2)}{sg(j.e3)}, "
                   f"S1+S2= {_f(r.e1s + r.e2s)} = {_f(r.e1s)}{sg(r.e2s)})")
    if r.zscore is not None:
        out.append(f"z-score: {_f(r.zscore[0])}, {_f(r.zscore[1])}")
    return "\n".join(out)


def predict(stage: ProbabilityStage, pairs: Sequence[Tuple[FastaRecord, FastaRecord]], opts: Optional[RpOpts] = None,
            ip_opts: Optional[RpIpOpts] = None, show_energy: bool = False, zscore: int = 0, num_shuffling: int = 1000,
            seed: int = 1, use_constraint: bool = False) -> List[PairResult]:
    """Joint structures of all `pairs`: one GPU batch for every pair's matrices, then the integer programmes on the
    host.  zscore in (1, 2, 12): per pair one more GPU batch with all its dinucleotide shuffles (the loop of
    src/ractip.cpp:1636-1657 with the probability work hoisted out of it).  use_constraint (-c): the records'
    structure lines constrain the pairs' probability matrices (constraint_line); shuffles have no structure line and
    stay unconstrained."""
    opts = opts if opts is not None else default_opts()
    ip_opts = ip_opts if ip_opts is not None else default_ip_opts()
    model: RpModel = stage.model
    energies = show_energy or zscore in (1, 2, 12)
    seqs = [(a.seq, b.seq) for a, b in pairs]
    cons = [(constraint_line(a), constraint_line(b)) for a, b in pairs] if use_constraint else None
    probs = stage.run_dense(seqs, opts, constraints=cons)
    out = []
    for (a, b), p in zip(pairs, probs):
        res = PairResult(a, b, solve_joint(model, a.seq, b.seq, p, ip_opts, energies=energies))
        if energies:
            _, _, res.e1s = solve_ss(model, a.seq, p.bp1, ip_opts, energy=True)
            _, _, res.e2s = solve_ss(model, b.seq, p.bp2, ip_opts, energy=True)
        if zscore in (1, 2, 12):
            r1, r2 = zscore_shuffles(a.seq, b.seq, num_shuffling, seed, zscore)
            sh = stage.run_dense(list(zip(r1, r2)), opts)
            rows = []
            for s1, s2, q in zip(r1, r2, sh):
                jp = solve_joint(model, s1, s2, q, ip_opts, energies=True)
                _, _, x1 = solve_ss(model, s1, q.bp1, ip_opts, energy=True)
                _, _, x2 = solve_ss(model, s2, q.bp2, ip_opts, energy=True)
                rows.append((jp.e1 + jp.e2 + jp.e3, x1 + x2))
            j = res.joint
            res.zscore = zscore_statistic(j.e1 + j.e2 + j.e3, res.e1s + res.e2s, rows)
        out.append(res)
    return out
