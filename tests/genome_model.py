"""Test helper: an independent byte model of a genome that is masked in place (mg_genome_mask, K5), read back
(mg_genome_fetch) and flagged (mg_genome_at_flags, K6), and of mask_from_gff (genome_tools.py:394-428).  It does not import
magot_b200, so it can be checked without a GPU.

Contigs are bytearrays.  A soft mask lower-cases A-Z only and a hard mask writes 'N', on 0-based half-open intervals that
are already clamped; upper_first upper-cases a-z only, everywhere, before the intervals are applied (Python 2 str.lower /
str.upper in the C locale, which is what bytes.lower / bytes.upper do).  The reverse complement is gencode_ref.revcomp:
acgtACGTnN- map as the reference maps them, every other byte becomes 'n'.

n_exceptions() is the size of the packed genome's side list of bytes that have no 4-bit code (include/magot_b200.h, K0):
a byte outside ACGTacgtNn-RYKM when it is packed, or an R/Y/K/M that a soft mask lower-cases.  A listed byte stays listed
when upper_first upper-cases it back to R/Y/K/M (its code does not change), and leaves the list when a hard mask overwrites
it.
"""
import numpy as np

import gencode_ref
import py2dict

ALPHABET = b"ACGTacgtNn-RYKM"
_IN_ALPHABET = np.zeros(256, dtype=bool)
_IN_ALPHABET[np.frombuffer(ALPHABET, dtype=np.uint8)] = True
_AT = np.zeros(256, dtype=np.uint8)
_AT[np.frombuffer(b"ATat", dtype=np.uint8)] = 1


def at_flags(seq):
    """1 where a byte of `seq` is one of "ATat", else 0 (position_dic.at_content, genome.py:1030-1034)."""
    return _AT[np.frombuffer(bytes(seq), dtype=np.uint8)]


class Genome(object):
    """Contigs as bytearrays plus, per base, whether the packed genome keeps it in its exception list."""

    def __init__(self, contigs):
        self.contigs = [bytearray(c) for c in contigs]
        self.listed = [~_IN_ALPHABET[np.frombuffer(bytes(c), dtype=np.uint8)] for c in self.contigs]

    def mask(self, contig, lo, hi, hard=False, upper_first=False):
        if upper_first:
            for c in self.contigs:
                c[:] = c.upper()
        for ci, a, b in zip(contig, lo, hi):
            ci, a, b = int(ci), int(a), int(b)
            assert 0 <= a <= b <= len(self.contigs[ci])
            c = self.contigs[ci]
            if hard:
                c[a:b] = b"N" * (b - a)
                self.listed[ci][a:b] = False
            else:
                c[a:b] = bytes(c[a:b]).lower()
                self.listed[ci][a:b] |= ~_IN_ALPHABET[np.frombuffer(bytes(c[a:b]), dtype=np.uint8)]

    def fetch(self, contig, lo, hi, minus=False):
        s = bytes(self.contigs[contig][lo:hi])
        return gencode_ref.revcomp(s) if minus else s

    def at_flags(self, contig, lo, hi):
        return at_flags(self.contigs[contig][lo:hi])

    def n_exceptions(self):
        return int(sum(int(x.sum()) for x in self.listed))

    def bytes_list(self):
        return [bytes(c) for c in self.contigs]


def _truth(option):
    if option in ("True", "T", "true", "t", "TRUE"):
        return True
    if option in ("False", "F", "false", "f", "FALSE"):
        return False
    raise ValueError(option)


def mask_from_gff(fasta_text, gff_text, mask_type="soft", overwrite_softmask="True", feature_type="CDS"):
    """The text mask_from_gff prints for FASTA bytes `fasta_text` and GFF text `gff_text` (str), as bytes.

    The seqid is the first word of a header; a repeated header starts that sequence over; CR bytes are dropped from
    sequence lines.  Every GFF line with more than 5 tabs whose third column is `feature_type` masks the list slice
    [start-1:stop] of its sequence under Python slice rules (start = 0 gives [-1:stop]).  A hard mask writes
    max(stop - start + 1, 0) 'N's into that slice; where the slice is shorter (clamped by the sequence end) the reference
    would change the sequence's length, and this model raises NotImplementedError instead, as the port does.  Records are
    printed in Python 2.7 dict order."""
    upper_first = _truth(overwrite_softmask)
    seqs = {}
    working = None
    lines = fasta_text.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    for line in lines:
        if line[:1] == b">":
            working = line.split()[0][1:].replace(b"\r", b"")
            seqs[working] = bytearray()
        elif line:
            seqs[working] += line.replace(b"\r", b"")
    if upper_first:
        for s in seqs.values():
            s[:] = s.upper()
    for line in gff_text.split("\n"):
        if line.count("\t") <= 5:
            continue
        fields = line.split("\t")
        if fields[2] != feature_type:
            continue
        seq = seqs[fields[0].encode("latin-1")]
        start, stop = int(fields[3]), int(fields[4])
        part = seq[start - 1:stop]
        if mask_type == "soft":
            seq[start - 1:stop] = bytes(part).lower()
        else:
            n = max(stop - start + 1, 0)
            if len(part) != n:
                raise NotImplementedError("%s:%d-%d" % (fields[0], start, stop))
            seq[start - 1:stop] = b"N" * n
    names = py2dict.py2_order(list(seqs))
    return b"".join(b">" + n + b"\n" + bytes(seqs[n]) + b"\n" for n in names)
