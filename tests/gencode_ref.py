"""Test helper: an independent statement of the NCBI genetic codes and a numpy restatement of Sequence.translate /
get_orfs / the six-frame ORF scan under any codon table.

The tables are rebuilt here from their published differences to table 1, not copied from magot_b200.gencode, so that
the two can be compared.  translate() follows magot_oracle.translate(library=...) (the reference's frame quirk, one
leading 'X' trimmed, lower case upper-cased, any codon with a base outside ACGT -> 'X'); sixframe() returns what
coracle.sixframe returns, for contigs far longer than the pure-Python oracle can take.
"""
import numpy as np

import magot_oracle as mo

STANDARD = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"   # NCBI table 1, codons in TCAG order
TCAG = "TCAG"

#: id -> {codon: residue} where the code differs from table 1 (NCBI's published tables)
DIFFS = {
    1: {}, 11: {},
    2: {"AGA": "*", "AGG": "*", "ATA": "M", "TGA": "W"},
    3: {"ATA": "M", "CTT": "T", "CTC": "T", "CTA": "T", "CTG": "T", "TGA": "W"},
    4: {"TGA": "W"},
    5: {"AGA": "S", "AGG": "S", "ATA": "M", "TGA": "W"},
    6: {"TAA": "Q", "TAG": "Q"},
    9: {"AAA": "N", "AGA": "S", "AGG": "S", "TGA": "W"},
    10: {"TGA": "C"},
    12: {"CTG": "S"},
    13: {"AGA": "G", "AGG": "G", "ATA": "M", "TGA": "W"},
    14: {"AAA": "N", "AGA": "S", "AGG": "S", "TAA": "Y", "TGA": "W"},
    16: {"TAG": "L"},
    21: {"AAA": "N", "AGA": "S", "AGG": "S", "ATA": "M", "TGA": "W"},
    22: {"TCA": "*", "TAG": "L"},
    23: {"TTA": "*"},
    24: {"AGA": "S", "AGG": "K", "TGA": "W"},
    25: {"TGA": "G"},
    26: {"CTG": "A"},
    29: {"TAA": "Y", "TAG": "Y"},
    30: {"TAA": "E", "TAG": "E"},
    33: {"TAA": "Y", "TGA": "W", "AGA": "S", "AGG": "K"},
}

#: id -> stop codons as listed with the tables
STOPS = {
    1: "TAA TAG TGA", 11: "TAA TAG TGA", 2: "TAA TAG AGA AGG", 3: "TAA TAG", 4: "TAA TAG", 5: "TAA TAG", 6: "TGA",
    9: "TAA TAG", 10: "TAA TAG", 12: "TAA TAG TGA", 13: "TAA TAG", 14: "TAG", 16: "TAA TGA", 21: "TAA TAG",
    22: "TCA TAA TGA", 23: "TTA TAA TAG TGA", 24: "TAA TAG", 25: "TAA TAG", 26: "TAA TAG TGA", 29: "TGA", 30: "TGA",
    33: "TAG",
}

#: one code per distinct stop set
STOP_SET_CODES = (1, 2, 3, 6, 14, 16, 22, 23)


def ncbi_string(code):
    """The code's 64 residues in NCBI (TCAG) order."""
    out = []
    for i, a in enumerate(STANDARD):
        c = TCAG[i >> 4] + TCAG[(i >> 2) & 3] + TCAG[i & 3]
        out.append(DIFFS[code].get(c, a))
    return "".join(out)


def library(code):
    s = ncbi_string(code)
    return {TCAG[i >> 4] + TCAG[(i >> 2) & 3] + TCAG[i & 3]: a for i, a in enumerate(s)}


def table64(code):
    """64 residues, index 16*b0 + 4*b1 + b2 with A=0 C=1 G=2 T=3."""
    lib = library(code)
    return "".join(lib["ACGT"[i >> 4] + "ACGT"[(i >> 2) & 3] + "ACGT"[i & 3]] for i in range(64))


_CODE = np.full(256, 4, dtype=np.int64)
for _i, _c in enumerate(b"ACGT"):
    _CODE[_c] = _i
    _CODE[_c + 32] = _i                                     # lower case
_COMP = np.full(256, ord("n"), dtype=np.uint8)             # genome.py:787: anything else -> 'n'
for _a, _b in zip(b"acgtACGTnN-", b"tgcaTGCAnN-"):
    _COMP[_a] = _b


def revcomp(seq):
    return _COMP[np.frombuffer(seq, dtype=np.uint8)[::-1]].tobytes()


def translate(seq, code_table, frame=0, minus=False, trimX=True):
    """Sequence.translate(library=...) of bytes `seq` under `code_table` (table64 string); None where the reference returns
    None.  Frames 1 and 2 start with the 1- / 2-base fragment, which no codon library holds: 'X'."""
    if minus:
        seq = revcomp(seq)
    n = len(seq)
    if not n > 2 + frame:
        return None
    c = _CODE[np.frombuffer(seq, dtype=np.uint8)]
    first = (0, 2, 4)[frame]
    m = max(0, (n - first) // 3)
    tri = c[first:first + 3 * m].reshape(m, 3)
    lut = np.frombuffer(code_table.encode() + b"X", dtype=np.uint8)
    idx = np.where((tri >= 4).any(axis=1), 64, tri[:, 0] * 16 + tri[:, 1] * 4 + tri[:, 2])
    out = lut[idx].tobytes()
    if frame:
        out = b"X" + out
    if trimX and out[:1] == b"X":
        out = out[1:]
    return out


def sixframe(seq, min_aa, code_table):
    """(residues back to back, [(frame, minus, start, len)]) -- coracle.sixframe under `code_table`."""
    aa, recs = [], []
    for frame in (0, 1, 2):
        for minus in (1, 0):
            t = translate(seq, code_table, frame, bool(minus))
            if not t:
                continue
            start = 0
            for part in t.split(b"*"):
                if len(part) >= min_aa:
                    aa.append(part)
                    recs.append((frame, minus, start, len(part)))
                start += len(part) + 1
    return b"".join(aa), recs


def get_orfs(seq, lib, longest=False, from_atg=False):
    """magot_oracle.get_orfs with translate(library=lib) (genome.py:824-851 under another code)."""
    orflist, candidate_list, longest_orf_len = [], [], 0
    for frame in (0, 1, 2):
        for st in ('-', '+'):
            t = mo.translate(seq, frame=frame, strand=st, library=lib)
            if t:
                for orf in t.split('*'):
                    output_orf = ('M' + ''.join(orf.split('M')[1:])) if from_atg else orf
                    if longest:
                        if len(output_orf) > longest_orf_len:
                            candidate_list.append(output_orf)
                            longest_orf_len = len(output_orf)
                    else:
                        orflist.append(output_orf)
    if longest:
        return candidate_list[-1]
    return orflist
