"""Variant consequences without a GPU: the VCF reader, the normalisation and the model variant_ref against hand-worked rows of
a two-exon gene on '+' and the same gene on '-', the phase skip, the genome_tools argument checks and the exported ABI."""
import gzip

import pytest

import gencode_ref as gref
import variant_ref as ref

VCF = b"".join(x.replace(b" ", b"\t") + b"\n" for x in (
    b"##fileformat=VCFv4.2",
    b"##contig=<ID=chr1>",
    b"#CHROM POS ID REF ALT QUAL FILTER INFO FORMAT S1",
    b"chr1 3 rs1 A C,g 50 PASS DP=3 GT 0/1",
    b"chr1 5 . GG G,<DEL>,* . . . GT 1/2",
    b"chr1 9 . g . . . .",
    b"chr1 10 bnd G G]chr2:5],.G,G. . . .",
    b"chr2 1 . C <INS> . . .",
))


def test_read_vcf_plain_and_gzip(tmp_path):
    from magot_b200 import variants
    for data in (VCF, gzip.compress(VCF)):
        p = tmp_path / "calls.vcf"
        p.write_bytes(data)
        for src in (str(p), data):
            v = variants.read_vcf(src)
            assert len(v) == 3
            assert v.chrom == ["chr1"] * 3 and v.pos.tolist() == [3, 3, 5] and v.ids == ["rs1", "rs1", "."]
            assert v.ref == [b"A", b"A", b"GG"] and v.alt == [b"C", b"g", b"G"]
            assert v.line.tolist() == [3, 3, 4] and v.alt_no.tolist() == [1, 2, 1]
            assert dict(v.skipped) == {"symbolic": 2, "star": 1, "missing": 1, "breakend": 3}
            assert len(v.lines) == 8 and v.lines[2].startswith(b"#CHROM")


def test_read_vcf_rejects_bad_lines():
    from magot_b200 import variants
    with pytest.raises(ValueError):
        variants.read_vcf(b"chr1\tx\t.\tA\tC\n")
    with pytest.raises(ValueError):
        variants.read_vcf(b"chr1\t5\t.\tA\n")


@pytest.mark.parametrize("pos, r, a, want", [
    (10, b"A", b"C", (10, 11, b"C")),                   # SNV
    (10, b"A", b"ATT", (11, 11, b"TT")),                # insertion with its anchor base
    (10, b"ATT", b"A", (11, 13, b"")),                  # deletion with its anchor base
    (10, b"AGGA", b"AGA", (11, 12, b"")),               # the suffix goes first: GGA / GA leave G, not the middle base
    (10, b"CAT", b"cgt", (11, 12, b"g")),               # an MNV framed by equal bases, case ignored
    (10, b"ATGC", b"AC", (11, 13, b"")),                # suffix C, then prefix A
    (10, b"TCA", b"GGTA", (10, 12, b"GGT")),            # complex: suffix A only
    (10, b"AAA", b"AAAA", (10, 10, b"A")),              # a repeat: the suffix strip moves the insertion to the start
])
def test_normalise(pos, r, a, want):
    assert ref.normalise(pos, r, a) == want


def _gene():
    """contig 0: CC | exon 1 ATGGCTTGGA | intron GTAAGTTTAG | exon 2 AAGTTTAAC | CCC, payload ATG GCT TGG AAA GTT TAA C;
    contig 1: its reverse complement, with the same gene on '-'."""
    from test_gpu_check import _table
    c0 = b"CC" + b"ATGGCTTGGA" + b"GTAAGTTTAG" + b"AAGTTTAAC" + b"CCC"
    c1 = gref.revcomp(c0)
    tbl = _table([[(0, 3, 12, 0), (0, 23, 31, 0)], [(1, 23, 32, 1), (1, 4, 12, 1)]])
    return [c0, c1], tbl


PLUS = [(0, 2, b"A", b"C"), (0, 9, b"G", b"A"), (0, 27, b"T", b"C"), (0, 5, b"G", b"N"), (0, 6, b"C", b"T"), (0, 7, b"T", b"C"),
        (0, 30, b"C", b"G"), (0, 4, b"GG", b"G"), (0, 6, b"C", b"CAAA"), (0, 23, b"AGTT", b"A"), (0, 13, b"T", b"C"),
        (0, 20, b"A", b"G"), (0, 30, b"CC", b"GA"), (0, 21, b"G", b"GT"), (0, 30, b"C", b"CA"), (0, 22, b"A", b"T")]
_COMP = {65: 84, 67: 71, 71: 67, 84: 65, 78: 78}
ALLELES = sorted(PLUS + [(1, 33 - p, bytes(_COMP[x] for x in r), bytes(_COMP[x] for x in a)) for _, p, r, a in PLUS
                         if len(r) == len(a) == 1], key=lambda x: (x[0], x[1]))

# (var, rec, seg, nuc_lo, nuc_hi, codon, cls, n_aff, ref_codon, alt_codon, ref_aa, alt_aa), worked out by hand from _gene()
ROWS = [
    (0, 0, 0, 0, 1, 0, 7, 1, 14, 30, b'M', b'L'),
    (1, 0, 0, 2, 3, 0, 4, 0, 255, 255, b'', b''),
    (2, 0, 0, 3, 4, 1, 10, 1, 39, 255, b'A', b'X'),
    (3, 0, 0, 4, 5, 1, 11, 1, 39, 47, b'A', b'V'),
    (4, 0, 0, 5, 5, 1, 5, 0, 255, 255, b'', b''),
    (5, 0, 0, 5, 6, 1, 12, 1, 39, 37, b'A', b'A'),
    (6, 0, 0, 7, 8, 2, 8, 1, 58, 50, b'W', b'*'),
    (7, 0, 0, -1, -1, -1, 2, 0, 255, 255, b'', b''),
    (8, 0, 0, -1, -1, -1, 1, 0, 255, 255, b'', b''),
    (9, 0, 0, -1, -1, -1, 1, 0, 255, 255, b'', b''),
    (10, 0, 1, 10, 11, 3, 11, 1, 0, 12, b'K', b'I'),
    (11, 0, 1, 12, 15, 4, 6, 0, 255, 255, b'', b''),
    (12, 0, 1, 15, 16, 5, 9, 1, 48, 16, b'*', b'Q'),
    (13, 0, 1, 18, 19, -1, 13, 0, 255, 255, b'', b''),
    (14, 0, 1, 18, 19, -1, 3, 0, 255, 255, b'', b''),
    (16, 1, 3, 18, 19, -1, 13, 0, 255, 255, b'', b''),
    (17, 1, 3, 15, 16, 5, 9, 1, 48, 16, b'*', b'Q'),
    (18, 1, 3, 10, 11, 3, 11, 1, 0, 12, b'K', b'I'),
    (19, 1, 2, -1, -1, -1, 1, 0, 255, 255, b'', b''),
    (20, 1, 2, -1, -1, -1, 2, 0, 255, 255, b'', b''),
    (21, 1, 2, 7, 8, 2, 8, 1, 58, 50, b'W', b'*'),
    (22, 1, 2, 5, 6, 1, 12, 1, 39, 37, b'A', b'A'),
    (23, 1, 2, 4, 5, 1, 11, 1, 39, 47, b'A', b'V'),
    (24, 1, 2, 3, 4, 1, 10, 1, 39, 255, b'A', b'X'),
    (25, 1, 2, 0, 1, 0, 7, 1, 14, 30, b'M', b'L'),
]


def test_model_against_hand_worked_rows():
    contigs, tbl = _gene()
    st, rows = ref.effects(contigs, tbl, ALLELES)
    assert st == [0] * len(ALLELES)
    assert [tuple(r[f] for f in ref.FIELDS) for r in rows] == ROWS
    assert {r[6] for r in ROWS} == set(range(1, 14))
    # the mirrored SNVs on '-' give the '+' classes, codons and residues
    plus = {(ALLELES[r[0]][1], ALLELES[r[0]][3]): r[5:] for r in ROWS if r[1] == 0}
    for r in ROWS:
        if r[1] == 1:
            _, p, rb, ab = ALLELES[r[0]]
            assert plus[(33 - p, bytes(_COMP[x] for x in ab))] == r[5:]


def test_model_phase_skip():
    from test_gpu_check import _table
    contigs, _ = _gene()
    tbl = _table([[(0, 3, 12, 0), (0, 23, 31, 0)], [(1, 23, 32, 1), (1, 4, 12, 1)]], [1, 0])
    _, rows = ref.effects(contigs, tbl, ALLELES, use_phase=True)
    got = {r["var"]: tuple(r[f] for f in ref.FIELDS) for r in rows if r["rec"] == 0}
    assert got[0] == (0, 0, 0, 0, 1, -1, 13, 0, 255, 255, b"", b"")         # payload 0 is the skipped base
    assert got[13] == (13, 0, 1, 18, 19, 5, 11, 1, 1, 2, b"N", b"K")       # payload 18 now ends codon 5: AAC -> AAG
    _, rows = ref.effects(contigs, tbl, ALLELES, use_phase=False)
    assert [r["cls"] for r in rows if r["var"] in (0, 13) and r["rec"] == 0] == [7, 13]


def test_model_status():
    contigs, tbl = _gene()
    cases = [(-1, 0, b"A", b"C"), (2, 0, b"A", b"C"), (0, -1, b"A", b"C"), (0, 33, b"CC", b"C"),
             (0, 2, b"T", b"C"), (0, 2, b"a", b"c"), (0, 2, b"", b"A"), (0, 2, b"A", b""), (0, 2, b"AT", b"at")]
    assert [ref.status(contigs, *c) for c in cases] == [1, 1, 1, 1, 2, 0, 3, 3, 3]
    assert ref.status([b"ACxT"], 0, 1, b"CX", b"C") == 2                    # an exception byte never matches


def test_tool_argument_errors(tmp_path):
    from magot_b200 import genome_tools
    for kw in (dict(genetic_code="7"), dict(start_codons="TAA"), dict(start_codons="AT"), dict(out_format="bed")):
        with pytest.raises(ValueError):
            genome_tools.variant_effects("missing.fa", "missing.gff", "missing.vcf", **kw)
    assert "variant_effects" in genome_tools.FUNCTIONS


def test_abi_exported():
    from magot_b200 import _lib, engine
    for name in ("mg_plan_variant_count", "mg_plan_variant_emit", "mg_plan_variant_emit_device"):
        assert name in _lib.SIGNATURES and getattr(_lib.lib, name)
    assert engine.VEF_DTYPE.itemsize == 64
    assert len(_lib.VEF_CLASSES) == 13 and _lib.VEF_CLASSES[10] == "MISSENSE"
