"""Test helper: an independent statement of the gene-model check (mg_plan_check, engine.Plan.check, AnnotationSet.check_cds,
genome_tools check_cds) in numpy / pure Python.

It works from host genome bytes (one bytes object per contig) and a RecordTable, applies the Python-slice clamp
contig[start-1:end] itself and does not import magot_b200.  Record r's payload is its clamped segments in emission order, each
reverse-complemented by its strand (gencode_ref.revcomp); codon i is payload[skip+3i : skip+3i+3].  Codon indices are
16*b0 + 4*b1 + b2 with A=0 C=1 G=2 T=3; 0xFF is an absent or ambiguous codon.  Codon tables come from gencode_ref.
"""
import numpy as np

import gencode_ref as gref

NO_START, NO_STOP, INTERNAL_STOP, PARTIAL_CODON, NONCANONICAL_SPLICE, AMBIGUOUS, EMPTY = (1 << k for k in range(7))
FIELDS = ("nuc_len", "gc", "n_codons", "n_ambig", "n_stop", "first_stop", "gc3", "n_junction", "n_noncanonical", "flags",
          "skip", "rem", "start_codon", "stop_codon")

_BASE = np.full(256, -1, dtype=np.int64)
for _i, _c in enumerate(b"ACGT"):
    _BASE[_c] = _i
    _BASE[ord(chr(_c).lower())] = _i


def clamp(L, start, end):
    """0-based [a, b) of contig[start-1:end] for a contig of L bases (Python slice semantics), b >= a."""
    a, b, _ = slice(int(start) - 1, int(end)).indices(L)
    return a, max(a, b)


def codon_index(codon):
    """Index of a 3-byte codon, or None when a base is outside A/C/G/T (either case)."""
    b = _BASE[np.frombuffer(bytes(codon), dtype=np.uint8)]
    if len(b) != 3 or (b < 0).any():
        return None
    return int(b[0] * 16 + b[1] * 4 + b[2])


def payload(contigs, tbl, r):
    out = []
    for e in range(int(tbl.rec_seg_off[r]), int(tbl.rec_seg_off[r + 1])):
        c = int(tbl.seg_contig[e])
        if c < 0 or c >= len(contigs):
            continue
        a, b = clamp(len(contigs[c]), tbl.seg_start[e], tbl.seg_end[e])
        s = contigs[c][a:b]
        out.append(gref.revcomp(s) if tbl.seg_strand[e] else s)
    return b"".join(out)


def _pair(contigs, c, lo, minus):
    """The dinucleotide read 5'->3' on the transcript strand: forward bases lo, lo+1, or the reverse complement of them."""
    s = contigs[c][lo:lo + 2]
    return gref.revcomp(s) if minus else s


def junction_class(contigs, tbl, e):
    """Class of the junction after segment e of tbl (0..4)."""
    r = int(np.searchsorted(tbl.rec_seg_off, e, side="right")) - 1
    if e + 1 >= int(tbl.rec_seg_off[r + 1]):
        return 0
    segs = []
    for k in (e, e + 1):
        c = int(tbl.seg_contig[k])
        if c < 0 or c >= len(contigs):
            return 0
        a, b = clamp(len(contigs[c]), tbl.seg_start[k], tbl.seg_end[k])
        if b <= a:
            return 0
        segs.append((c, a, b, bool(tbl.seg_strand[k])))
    (c0, a0, b0, m0), (c1, a1, b1, m1) = segs
    if c0 != c1 or m0 != m1:
        return 0
    if not m0:
        if a1 - b0 < 4:
            return 0
        donor, acceptor = contigs[c0][b0:b0 + 2], contigs[c0][a1 - 2:a1]
    else:
        if a0 - b1 < 4:
            return 0
        donor, acceptor = _pair(contigs, c0, a0 - 2, True), _pair(contigs, c0, b1, True)
    d, x = donor.upper(), acceptor.upper()
    if d == b"GT" and x == b"AG":
        return 1
    if d == b"GC" and x == b"AG":
        return 2
    if d == b"AT" and x == b"AC":
        return 3
    return 4


def check(contigs, tbl, code=1, starts=("ATG",), use_phase=False):
    """(records: list of dicts with FIELDS, counts: int64 [n_rec, 64], junctions: int8 [n_seg]) for every record of tbl."""
    table = gref.table64(code)
    stop = [a == "*" for a in table]
    start = set(codon_index(c.upper().encode()) for c in starts)
    junc = np.array([junction_class(contigs, tbl, e) for e in range(tbl.n_seg)], dtype=np.int8)
    recs, counts = [], np.zeros((tbl.n_rec, 64), dtype=np.int64)
    for r in range(tbl.n_rec):
        s = payload(contigs, tbl, r)
        skip = 0
        if use_phase and tbl.rec_phase is not None and 0 <= int(tbl.rec_phase[r]) <= 2:
            skip = int(tbl.rec_phase[r])
        L = len(s) - skip
        n = L // 3 if L > 0 else 0
        rem = L % 3 if L > 0 else 0
        idx = [codon_index(s[skip + 3 * i:skip + 3 * i + 3]) for i in range(n)]
        stops = [i for i, c in enumerate(idx) if c is not None and stop[c]]
        gc = gc3 = 0
        for c in idx:
            if c is None:
                continue
            counts[r, c] += 1
            bases = (c >> 4, (c >> 2) & 3, c & 3)
            gc += sum(1 for b in bases if b in (1, 2))
            gc3 += bases[2] in (1, 2)
        sc = idx[0] if n and idx[0] is not None else 0xFF
        ec = idx[-1] if n and idx[-1] is not None else 0xFF
        terminal = bool(n) and idx[-1] is not None and stop[idx[-1]]
        j = junc[int(tbl.rec_seg_off[r]):int(tbl.rec_seg_off[r + 1])]
        flags = 0
        if sc == 0xFF or sc not in start:
            flags |= NO_START
        if not terminal:
            flags |= NO_STOP
        if len(stops) - terminal > 0:
            flags |= INTERNAL_STOP
        if rem:
            flags |= PARTIAL_CODON
        if (j == 4).any():
            flags |= NONCANONICAL_SPLICE
        n_ambig = sum(1 for c in idx if c is None)
        if n_ambig:
            flags |= AMBIGUOUS
        if n == 0:
            flags |= EMPTY
        recs.append(dict(nuc_len=len(s), gc=gc, n_codons=n, n_ambig=n_ambig, n_stop=len(stops),
                         first_stop=stops[0] if stops else -1, gc3=gc3, n_junction=int((j > 0).sum()),
                         n_noncanonical=int((j == 4).sum()), flags=flags, skip=skip, rem=rem, start_codon=sc, stop_codon=ec))
    return recs, counts, junc


def compare(got, want):
    """Field-by-field comparison of a CHECK_DTYPE array with check()'s records; returns the first mismatch or None."""
    if len(got) != len(want):
        return "%d records, want %d" % (len(got), len(want))
    for r, w in enumerate(want):
        for f in FIELDS:
            if int(got[f][r]) != w[f]:
                return "record %d field %s: %d, want %d" % (r, f, int(got[f][r]), w[f])
    return None
