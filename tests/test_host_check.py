"""The gene-model check without a GPU: the model cdscheck_ref on hand-written gene models (a good gene, an internal stop, no
start, no stop, rem 1 and 2, phase 1 and 2, ambiguous codons, every junction class on both strands, a 3-base gap and segments
out of order), gc / gc3 against the 64 counts, the argument checks of genome_tools check_cds, and its two text formats built
from given arrays."""
import numpy as np
import pytest

import cdscheck_ref as ref
import gencode_ref as gref

#   exon 1      intron GT..AG      exon 2
GOOD = b"ATGAAACCC" + b"GTAAAG" + b"GGGTTTTAA"


def _table(segs, phase=None):
    from magot_b200.tables import RecordTable
    rec_off = np.concatenate(([0], np.cumsum([len(r) for r in segs])))
    flat = [x for r in segs for x in r]
    cols = [np.array([x[k] for x in flat], dtype=t) for k, t in enumerate((np.int32, np.int64, np.int64, np.int8))]
    n = len(segs)
    z = np.zeros(n, dtype=np.int32)
    return RecordTable(rec_off, *cols, np.zeros(n, np.int64), z, z, np.zeros(0, np.uint8),
                       None if phase is None else np.array(phase, dtype=np.int8))


def _one(contig, segs, phase=None, use_phase=False, code=1, starts=("ATG",)):
    recs, counts, junc = ref.check([contig], _table([segs], None if phase is None else [phase]), code, starts, use_phase)
    return recs[0], counts[0], junc


def _names(flags):
    return {n for k, n in enumerate(("NO_START", "NO_STOP", "INTERNAL_STOP", "PARTIAL_CODON", "NONCANONICAL_SPLICE",
                                     "AMBIGUOUS", "EMPTY")) if flags >> k & 1}


def test_good_gene_plus_and_minus():
    r, c, j = _one(GOOD, [(0, 1, 9, 0), (0, 16, 24, 0)])
    assert r["flags"] == 0 and r["n_codons"] == 6 and r["n_stop"] == 1 and r["first_stop"] == 5
    assert r["start_codon"] == ref.codon_index(b"ATG") and r["stop_codon"] == ref.codon_index(b"TAA")
    assert list(j) == [1, 0] and r["n_junction"] == 1 and r["n_noncanonical"] == 0
    rc = gref.revcomp(GOOD)
    L = len(rc)
    r, c, j = _one(rc, [(0, L - 8, L, 1), (0, L - 23, L - 15, 1)])
    assert r["flags"] == 0 and list(j) == [1, 0]


def test_internal_stop_no_start_no_stop_partial():
    r, _, _ = _one(b"ATGTAGAAATAA", [(0, 1, 12, 0)])
    assert _names(r["flags"]) == {"INTERNAL_STOP"} and r["first_stop"] == 1 and r["n_stop"] == 2
    r, _, _ = _one(b"CTGAAATAA", [(0, 1, 9, 0)])
    assert _names(r["flags"]) == {"NO_START"}
    r, _, _ = _one(b"ATGAAAAAA", [(0, 1, 9, 0)])
    assert _names(r["flags"]) == {"NO_STOP"} and r["first_stop"] == -1
    r, _, _ = _one(b"ATGAAATAAC", [(0, 1, 10, 0)])
    assert _names(r["flags"]) == {"PARTIAL_CODON"} and r["rem"] == 1 and r["stop_codon"] == ref.codon_index(b"TAA")
    r, _, _ = _one(b"ATGAAATAACC", [(0, 1, 11, 0)])
    assert r["rem"] == 2 and "PARTIAL_CODON" in _names(r["flags"])
    r, _, _ = _one(b"AT", [(0, 1, 2, 0)])
    assert _names(r["flags"]) == {"EMPTY", "NO_START", "NO_STOP", "PARTIAL_CODON"} and r["start_codon"] == 0xFF


def test_phase_and_ambiguous():
    seq = b"CCATGAAATAA"
    for ph, skip in ((1, 1), (2, 2), (0, 0), (3, 0), (-1, 0)):
        r, _, _ = _one(seq, [(0, 1, 11, 0)], phase=ph, use_phase=True)
        assert r["skip"] == skip
    r, _, _ = _one(seq, [(0, 1, 11, 0)], phase=2, use_phase=True)
    assert r["flags"] == 0 and r["n_codons"] == 3
    r, _, _ = _one(seq, [(0, 1, 11, 0)], phase=2, use_phase=False)
    assert r["skip"] == 0 and "NO_START" in _names(r["flags"])
    r, c, _ = _one(b"ATGNNNaaRtaa", [(0, 1, 12, 0)])
    assert r["n_ambig"] == 2 and _names(r["flags"]) == {"AMBIGUOUS"} and int(c.sum()) == 2
    r, _, _ = _one(b"ATGAAATAN", [(0, 1, 9, 0)])
    assert r["stop_codon"] == 0xFF and "NO_STOP" in _names(r["flags"])


@pytest.mark.parametrize("donor,acceptor,cls", [(b"GT", b"AG", 1), (b"GC", b"AG", 2), (b"AT", b"AC", 3), (b"GT", b"AC", 4),
                                                (b"gt", b"ag", 1), (b"GN", b"AG", 4), (b"CT", b"AG", 4)])
def test_junction_classes_both_strands(donor, acceptor, cls):
    contig = b"ATGAAA" + donor + b"CCCC" + acceptor + b"TTTTAA"
    r, _, j = _one(contig, [(0, 1, 6, 0), (0, 15, 20, 0)])
    assert list(j) == [cls, 0] and r["n_junction"] == 1 and r["n_noncanonical"] == (cls == 4)
    assert ("NONCANONICAL_SPLICE" in _names(r["flags"])) == (cls == 4)
    rc = gref.revcomp(contig)
    L = len(rc)
    _, _, j = _one(rc, [(0, L - 5, L, 1), (0, L - 19, L - 14, 1)])
    assert list(j) == [cls, 0]


def test_no_junction_cases():
    c = b"ATGAAAGTCCCAGTTTTAA" * 2
    assert list(_one(c, [(0, 1, 6, 0), (0, 10, 20, 0)])[2]) == [0, 0]           # a 3-base gap
    assert list(_one(c, [(0, 1, 6, 0), (0, 11, 20, 0)])[2]) == [4, 0]           # 4 bases: a junction
    assert list(_one(c, [(0, 11, 20, 0), (0, 1, 6, 0)])[2]) == [0, 0]           # out of order
    assert list(_one(c, [(0, 1, 12, 0), (0, 10, 20, 0)])[2]) == [0, 0]          # overlap
    assert list(_one(c, [(0, 1, 6, 0), (0, 11, 20, 1)])[2]) == [0, 0]           # strand change
    assert list(_one(c, [(0, 1, 6, 0), (0, 80, 90, 0), (0, 11, 20, 0)])[2]) == [0, 0, 0]   # clamped-away segment
    assert list(_one(c, [(0, 1, 6, 0), (0, -20, -10, 0)])[2]) == [4, 0]         # negative coordinates: Python slice rules


def test_gc_from_counts():
    rng = np.random.default_rng(1)
    contig = np.frombuffer(b"ACGTacgtN", dtype=np.uint8)[rng.integers(0, 9, size=5000)].tobytes()
    segs = [[(0, int(a), int(a) + int(rng.integers(0, 300)), int(rng.integers(0, 2)))] for a in rng.integers(1, 4500, size=200)]
    recs, counts, _ = ref.check([contig], _table(segs))
    idx = np.arange(64)
    b = np.stack([idx >> 4, (idx >> 2) & 3, idx & 3])
    gcb = ((b == 1) | (b == 2)).sum(axis=0)
    for r, row in zip(recs, counts):
        assert r["gc"] == int((row * gcb).sum())
        assert r["gc3"] == int((row * ((b[2] == 1) | (b[2] == 2))).sum())
        assert int(row.sum()) == r["n_codons"] - r["n_ambig"]


def test_tool_argument_errors(tmp_path):
    from magot_b200 import genome_tools
    missing = str(tmp_path / "missing.fa")
    with pytest.raises(ValueError, match="genetic_code"):
        genome_tools.check_cds(missing, missing, genetic_code="7")
    with pytest.raises(ValueError, match="out_format"):
        genome_tools.check_cds(missing, missing, out_format="gff3")
    with pytest.raises(ValueError, match="stop codon"):
        genome_tools.check_cds(missing, missing, start_codons="ATG,TGA")
    with pytest.raises(ValueError, match="A/C/G/T"):
        genome_tools.check_cds(missing, missing, start_codons="AUG")
    with pytest.raises(NameError):
        genome_tools.check_cds(missing, missing, use_phase="yes")
    with pytest.raises(NameError):
        genome_tools.check_cds(missing, missing, only_ok="1")


def _recs(rows):
    from magot_b200 import engine
    a = np.zeros(len(rows), dtype=engine.CHECK_DTYPE)
    for i, row in enumerate(rows):
        for k, v in row.items():
            a[k][i] = v
    return a


def test_tsv_text():
    from magot_b200 import genome_tools
    recs = _recs([dict(nuc_len=24, gc=7, n_codons=8, n_stop=1, first_stop=7, gc3=3, n_junction=1, flags=0, start_codon=14,
                       stop_codon=48),
                  dict(nuc_len=13, gc=2, n_codons=4, n_ambig=1, n_stop=2, first_stop=1, gc3=0, n_junction=2, n_noncanonical=1,
                       flags=4 | 8 | 16 | 32 | 1, skip=1, rem=0, start_codon=0xFF, stop_codon=50),
                  dict(nuc_len=2, n_codons=0, flags=1 | 2 | 8 | 64, rem=2, start_codon=0xFF, stop_codon=0xFF)])
    lines = genome_tools._check_tsv_lines(["g1", "g2", "g3"], recs)
    assert lines == [
        "#ID\tnuc_len\tcodons\tskip\trem\tstart\tstop\tinternal_stops\tfirst_internal_stop\tambiguous\tgc\tgc3\tjunctions\t"
        "noncanonical\tstatus",
        "g1\t24\t8\t0\t0\tATG\tTAA\t0\t.\t0\t0.2917\t0.3750\t1\t0\tok",
        "g2\t13\t4\t1\t0\t.\tTAG\t1\t1\t1\t0.2222\t0.0000\t2\t1\tNO_START,INTERNAL_STOP,PARTIAL_CODON,NONCANONICAL_SPLICE,AMBIGUOUS",
        "g3\t2\t0\t0\t2\t.\t.\t0\t.\t0\t.\t.\t0\t0\tNO_START,NO_STOP,PARTIAL_CODON,EMPTY"]


def test_codon_usage_text():
    from magot_b200 import genome_tools
    counts = np.zeros(64, dtype=np.int64)
    counts[ref.codon_index(b"ATG")] = 6
    counts[ref.codon_index(b"TTT")] = 3
    counts[ref.codon_index(b"TTC")] = 1
    lines = genome_tools._codon_usage_lines(counts, 1)
    assert len(lines) == 65 and lines[0] == "#codon\tresidue\tcount\tper_thousand\tfraction"
    assert lines[1] == "TTT\tF\t3\t300.00\t0.7500"
    assert lines[2] == "TTC\tF\t1\t100.00\t0.2500"
    assert lines[3] == "TTA\tL\t0\t0.00\t."
    assert lines[11] == "TAA\t*\t0\t0.00\t."
    assert lines[1 + 35] == "ATG\tM\t6\t600.00\t1.0000"
    assert [x.split("\t")[0] for x in lines[1:5]] == ["TTT", "TTC", "TTA", "TTG"]
    assert genome_tools._codon_usage_lines(np.zeros(64), 2)[15].split("\t")[1:] == ["W", "0", ".", "."]   # TGA is W in table 2
    assert ".".join(lines).count("\t") == 4 * 65
