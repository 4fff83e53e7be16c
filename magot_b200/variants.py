"""VCF input for AnnotationSet.variant_effects and `genome_tools variant_effects`: one allele per ALT of each data line.

A Python line loop: VCF files of an annotation pipeline are read once, and the device join and classification
(mg_plan_variant_count / _emit) do the per-allele work.  Genotype columns are not read.
"""
import collections
import gzip

import numpy as np

#: reasons an ALT is not turned into an allele
SKIP_REASONS = ("symbolic", "star", "missing", "breakend")


class VcfAlleles(object):
    """Alleles of a VCF, in line order then ALT order.  Per allele: line (index into `lines`), alt_no (1-based ALT number),
    chrom, pos (1-based VCF POS), id, ref, alt (bytes).  `lines` holds every input line without its line end (header lines
    included); `skipped` counts the ALTs left out per reason (SKIP_REASONS)."""

    def __init__(self, lines, line, alt_no, chrom, pos, ids, ref, alt, skipped):
        self.lines = lines
        self.line = np.asarray(line, dtype=np.int64)
        self.alt_no = np.asarray(alt_no, dtype=np.int32)
        self.chrom, self.ids, self.ref, self.alt = chrom, ids, ref, alt
        self.pos = np.asarray(pos, dtype=np.int64)
        self.skipped = skipped

    def __len__(self):
        return len(self.chrom)


def _skip_reason(alt):
    if alt.startswith(b"<"):
        return "symbolic"
    if alt == b"*":
        return "star"
    if alt == b"." or not alt:
        return "missing"
    if b"[" in alt or b"]" in alt or alt.startswith(b".") or alt.endswith(b"."):
        return "breakend"
    return None


def read_vcf(path_or_bytes):
    """VcfAlleles of a VCF given as a path (plain or gzip / BGZF, detected from the magic bytes) or as its bytes."""
    if isinstance(path_or_bytes, (bytes, bytearray, memoryview)):
        data = bytes(path_or_bytes)
    else:
        with open(path_or_bytes, "rb") as f:
            data = f.read()
    if data[:2] == b"\x1f\x8b":
        data = gzip.decompress(data)
    lines = data.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    lines = [x[:-1] if x.endswith(b"\r") else x for x in lines]
    line, alt_no, chrom, pos, ids, ref, alt = [], [], [], [], [], [], []
    skipped = collections.OrderedDict((k, 0) for k in SKIP_REASONS)
    for k, text in enumerate(lines):
        if not text or text.startswith(b"#"):
            continue
        cols = text.split(b"\t")
        if len(cols) < 5:
            raise ValueError("VCF line %d has %d columns, at least 5 are needed" % (k + 1, len(cols)))
        try:
            p = int(cols[1])
        except ValueError:
            raise ValueError("VCF line %d: POS %r is not an integer" % (k + 1, cols[1].decode("latin-1")))
        for n, a in enumerate(cols[4].split(b","), 1):
            why = _skip_reason(a)
            if why:
                skipped[why] += 1
                continue
            line.append(k)
            alt_no.append(n)
            chrom.append(cols[0].decode("latin-1"))
            pos.append(p)
            ids.append(cols[2].decode("latin-1"))
            ref.append(cols[3])
            alt.append(a)
    return VcfAlleles(lines, line, alt_no, chrom, pos, ids, ref, alt, skipped)
