"""Start-to-stop ORF calling without a GPU: hand-written cases for the test reference (orfcall_ref), gencode.start64's
argument checks and call_orfs' text output (order, IDs, the partial tag) from records built here."""
import numpy as np
import pytest

import gencode_ref as gref
import orfcall_ref as ref


def _all(seq, min_aa=0, code=1, starts=("ATG",), partial=False):
    recs, aa = ref.call_list([seq], [0], min_aa, code, starts, partial)
    return [(r[1], r[2], r[3], r[5], r[6], aa[r[8]:r[8] + r[7]].decode()) for r in recs]


ATG = ref.codon_index("ATG")


def test_atg_to_stop():
    assert _all(b"ATGAAATAG") == [(0, 0, 0, 0, 9, "MK")]
    recs, aa = ref.call_list([b"ATGAAATAG"], [0], 0)
    assert recs == [(0, 0, 0, 0, ATG, 0, 9, 2, 0)] and aa == b"MK"


def test_reverse_complement_gives_the_orf_on_minus():
    assert _all(gref.revcomp(b"ATGAAATAG")) == [(1, 0, 0, 0, 9, "MK")]


def test_phase_one_and_last_codons():
    assert _all(b"CATGAAATAGC") == [(0, 1, 0, 1, 10, "MK")]
    assert _all(gref.revcomp(b"CATGAAATAGC")) == [(1, 1, 0, 1, 10, "MK")]
    # a start at the last codon of each strand: a one-residue 3' partial
    assert _all(b"AAAATG", partial=True) == [(0, 0, 1, 3, 6, "M")]
    assert _all(b"CATTTT", partial=True) == [(1, 0, 1, 0, 3, "M")]
    assert _all(b"AAAATG") == [] and _all(b"CATTTT") == []


def test_adjacent_stops_and_no_start():
    assert _all(b"TAATAGTGA", partial=True) == []
    assert _all(b"ATGTAATAG") == [(0, 0, 0, 0, 6, "M")]
    assert _all(b"AAATTTTAG", partial=True) == []


def test_three_prime_partial():
    assert _all(b"ATGAAAAAA") == []
    assert _all(b"ATGAAAAAA", partial=True) == [(0, 0, 1, 0, 9, "MKK")]
    assert _all(b"ATGAAAAAA", min_aa=4, partial=True) == []


def test_alternative_start_is_read_as_m():
    assert _all(b"GTGAAATAG") == []
    recs, aa = ref.call_list([b"GTGAAATAG"], [0], 0, starts=("ATG", "GTG", "TTG"))
    assert aa == b"MK" and recs[0][4] == ref.codon_index("GTG")


def test_nested_starts_give_one_orf():
    assert _all(b"ATGATGAAATAG") == [(0, 0, 0, 0, 12, "MMK")]


def test_case_and_non_acgt():
    assert _all(b"atgaaatag") == [(0, 0, 0, 0, 9, "MK")]
    assert _all(b"ATGANATAG") == [(0, 0, 0, 0, 9, "MX")]
    assert _all(b"ANGAAATAG", partial=True) == []
    assert _all(b"ATGAAATNG", partial=True) == [(0, 0, 1, 0, 9, "MKX")]    # TNG is no stop


def test_short_contigs():
    for n in range(6):
        assert _all(b"ATGATG"[:n], partial=True) == ([] if n < 3 else [(0, 0, 1, 0, 3, "M")])
        assert _all(b"NNNNN"[:n], partial=True) == []


def test_min_aa_counts_m_and_excludes_the_stop():
    assert _all(b"ATGAAATAG", min_aa=2) == [(0, 0, 0, 0, 9, "MK")]
    assert _all(b"ATGAAATAG", min_aa=3) == []


def test_other_code():
    # table 2: AGA is a stop, TGA is W
    assert _all(b"ATGTGAAGA", code=2) == [(0, 0, 0, 0, 9, "MW")]


def test_start64_validation():
    from magot_b200 import gencode
    t = gencode.start64(["ATG"])
    assert len(t) == 64 and t[ATG] == 1 and sum(t) == 1
    t = gencode.start64(("atg", "GTG", "TTG"), 11)
    assert sum(t) == 3 and t[ref.codon_index("TTG")] == 1
    assert gencode.start64("ATG") == gencode.start64(["ATG"])
    for bad in ([], ["AT"], ["ATGA"], ["ANG"], ["AUG"], ["TAA"]):
        with pytest.raises(ValueError):
            gencode.start64(bad)
    with pytest.raises(ValueError):
        gencode.start64(["AGA"], 2)                          # a stop of table 2
    gencode.start64(["AGA"], 1)
    with pytest.raises(ValueError):
        gencode.start64(["ATG"], 7)                          # unsupported table


def _recs(rows):
    from magot_b200 import orfs
    a = np.zeros(len(rows), dtype=orfs.ORFCALL_DTYPE)
    for i, (c, minus, phase, flags, sc, lo, hi, n) in enumerate(rows):
        a[i] = (c, minus, phase, flags, sc, lo, hi, n, 0)
    return a


def test_text_output():
    from magot_b200 import genome_tools as gt
    gtg = ref.codon_index("GTG")
    rows = [(5, 1, 0, 0, ATG, 100, 400, 99), (5, 0, 2, 1, gtg, 100, 200, 33), (5, 0, 0, 0, ATG, 100, 403, 100),
            (2, 0, 1, 0, ATG, 7, 310, 100), (5, 0, 1, 0, ATG, 40, 343, 100)]
    recs = _recs(rows)
    order = gt._orf_order([5, 2], recs)
    assert order.tolist() == [4, 2, 1, 0, 3]
    s = recs[order]
    names = {5: "chrA", 2: "scaf 2"}
    lines = gt._orf_lines(names, s, "gff3")
    assert lines == ["##gff-version 3",
                     "chrA\tmagot_b200\tORF\t41\t343\t.\t+\t.\tID=chrA_orf1;start_codon=ATG",
                     "chrA\tmagot_b200\tORF\t101\t403\t.\t+\t.\tID=chrA_orf2;start_codon=ATG",
                     "chrA\tmagot_b200\tORF\t101\t200\t.\t+\t.\tID=chrA_orf3;start_codon=GTG;partial=3prime",
                     "chrA\tmagot_b200\tORF\t101\t400\t.\t-\t.\tID=chrA_orf4;start_codon=ATG",
                     "scaf 2\tmagot_b200\tORF\t8\t310\t.\t+\t.\tID=scaf 2_orf1;start_codon=ATG"]
    seqs = ["P%d" % i for i in range(5)]
    assert gt._orf_lines(names, s, "protein", seqs)[:4] == [">chrA_orf1 chrA:41-343(+)", "P0", ">chrA_orf2 chrA:101-403(+)", "P1"]
    assert gt._orf_lines(names, s, "nucleotide", seqs)[-2:] == [">scaf 2_orf1 scaf 2:8-310(+)", "P4"]


def test_reference_cli_order_matches_the_tool():
    from magot_b200 import genome_tools as gt
    rng = np.random.default_rng(3)
    contigs = [rng.choice(np.frombuffer(b"ACGTacgtN", dtype=np.uint8), size=n).tobytes() for n in (3000, 500, 7)]
    ids = [2, 0, 1]
    recs, _ = ref.call_list(contigs, ids, 5, starts=("ATG", "CTG"), partial=True)
    assert recs
    a = _recs([r[:8] for r in recs])
    assert gt._orf_order(ids, a).tolist() == ref.cli_order(recs)


def test_call_orfs_rejects_bad_arguments_before_device_work(tmp_path):
    from magot_b200 import genome_tools as gt
    fa = tmp_path / "g.fa"
    fa.write_text(">a\nATGAAATAG\n")
    with pytest.raises(ValueError):
        gt.call_orfs(str(fa), out_format="bed")
    with pytest.raises(ValueError):
        gt.call_orfs(str(fa), start_codons="TAA")
    with pytest.raises(ValueError):
        gt.call_orfs(str(fa), genetic_code="27")
    assert "call_orfs" in gt.FUNCTIONS
