"""Test helper: an independent numpy statement of start-to-stop ORF calling (mg_orfcall_count, orfs.call_orfs,
genome_tools call_orfs).

For each strand (minus = the reverse complement) and true phase p, codons start at offset p + 3k of the strand's 5'->3'
sequence.  Lower case is upper case; a codon with a base outside ACGT is neither a start nor a stop (gencode_ref._CODE).
Every stretch between two stops (or a contig end) yields at most one ORF: from its first start codon through the stop that
ends it; one that reaches the contig end without a stop is a 3' partial.  The protein runs from the start codon up to, not
including, the stop, with 'M' first.  Codon tables come from gencode_ref, not from magot_b200.gencode.
"""
import numpy as np

import gencode_ref as gref

#: K4's stream order: frames 0, 1, 2 read residue classes 0, 2, 1; minus before plus
ABI_STREAMS = [(phase, minus) for phase in (0, 2, 1) for minus in (1, 0)]


def codon_index(codon):
    """16*b0 + 4*b1 + b2 with A=0 C=1 G=2 T=3."""
    return "ACGT".index(codon[0]) * 16 + "ACGT".index(codon[1]) * 4 + "ACGT".index(codon[2])


def _flags(codons):
    f = np.zeros(65, dtype=bool)                             # index 64: a codon with a base outside ACGT
    for c in codons:
        f[codon_index(c.upper())] = True
    return f


def stream_orfs(seq, minus, phase, min_aa, code, starts=("ATG",), partial=False):
    """ORFs of one strand and phase of bytes `seq`, in ascending order of their start on that strand: a list of
    (flags, start_codon, lo, hi, len, protein bytes)."""
    L = len(seq)
    s = gref.revcomp(seq) if minus else seq
    c = gref._CODE[np.frombuffer(s, dtype=np.uint8)]
    m = (L - phase) // 3 if L > phase else 0
    if m == 0:
        return []
    tri = c[phase:phase + 3 * m].reshape(m, 3)
    idx = np.where((tri >= 4).any(axis=1), 64, tri[:, 0] * 16 + tri[:, 1] * 4 + tri[:, 2])
    table = gref.table64(code)
    stop_f = np.array([a == "*" for a in table] + [False])
    start_f = _flags(starts)
    stops = np.flatnonzero(stop_f[idx])
    first = np.flatnonzero(start_f[idx])
    seg = np.searchsorted(stops, first, side="right")        # stretch of each start: the number of stops before it
    _, keep = np.unique(seg, return_index=True)              # the first start of each stretch
    lut = np.frombuffer(table.encode() + b"X", dtype=np.uint8)
    out = []
    for k in first[keep]:
        j = int(np.searchsorted(stops, k))
        stop = j < stops.size
        n = int(stops[j] - k) if stop else m - int(k)
        if n < min_aa or not (stop or partial):
            continue
        q = phase + 3 * int(k)
        span = 3 * n + (3 if stop else 0)
        lo = L - q - span if minus else q
        prot = b"M" + lut[idx[k + 1:k + n]].tobytes()
        out.append((0 if stop else 1, int(idx[k]), lo, lo + span, n, prot))
    return out


def call_list(contigs, ids, min_aa, code=1, starts=("ATG",), partial=False):
    """ORFs of contigs[ids] in the ABI's order (contig in list order, stream in ABI_STREAMS order, position on the strand).
    Returns (records: list of (contig, minus, phase, flags, start_codon, lo, hi, len, aa_off), residues: bytes)."""
    recs, aa, off = [], [], 0
    for ci in ids:
        for phase, minus in ABI_STREAMS:
            for flags, sc, lo, hi, n, prot in stream_orfs(contigs[ci], minus, phase, min_aa, code, starts, partial):
                recs.append((ci, minus, phase, flags, sc, lo, hi, n, off))
                aa.append(prot)
                off += n
    return recs, b"".join(aa)


def cli_order(recs):
    """Indices of ABI-ordered records in call_orfs' order: contig blocks kept, then lo, '+' before '-', then phase."""
    blocks, pos = {}, []
    for i, r in enumerate(recs):
        pos.append(blocks.setdefault(r[0], len(blocks)))
    return sorted(range(len(recs)), key=lambda i: (pos[i], recs[i][5], recs[i][1], recs[i][2], i))


def cli_lines(contigs, names, ids, min_aa, code, starts, partial, out_format):
    """The text lines genome_tools call_orfs prints for contigs[ids] (names[ci] = seqid), built from this reference."""
    recs, aa = call_list(contigs, ids, min_aa, code, starts, partial)
    lines = ["##gff-version 3"] if out_format == "gff3" else []
    count = {}
    for i in cli_order(recs):
        ci, minus, phase, flags, sc, lo, hi, n, off = recs[i]
        count[ci] = count.get(ci, 0) + 1
        oid = "%s_orf%d" % (names[ci], count[ci])
        strand = "-" if minus else "+"
        if out_format == "gff3":
            attrs = "ID=%s;start_codon=%s" % (oid, "ACGT"[sc >> 4] + "ACGT"[(sc >> 2) & 3] + "ACGT"[sc & 3])
            if flags & 1:
                attrs += ";partial=3prime"
            lines.append("\t".join((names[ci], "magot_b200", "ORF", str(lo + 1), str(hi), ".", strand, ".", attrs)))
            continue
        lines.append(">%s %s:%d-%d(%s)" % (oid, names[ci], lo + 1, hi, strand))
        if out_format == "protein":
            lines.append(aa[off:off + n].decode())
        else:
            nuc = contigs[ci][lo:hi]
            lines.append((gref.revcomp(nuc) if minus else nuc).decode("latin-1"))
    return lines
