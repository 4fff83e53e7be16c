"""The CDS prediction without a GPU: the model cdspredict_ref on hand-written payloads (a stop at the very end, no stop, a start
at a frame's first codon with and without the 5' partial flag, a stretch that is only a stop, min_aa around n_aa, ties across
frames, ambiguous and lower-case codons), the model against a plain codon-by-codon walk under five genetic codes and three start
sets, the mapping of ORFs back to '+' and '-' segments (clamped-away, empty and negative ones) with their phases, the antisense
table, the three text formats of genome_tools predict_cds built from model results, and its argument checks."""
import numpy as np
import pytest

import cdscheck_ref as cref
import cdspredict_ref as ref
import gencode_ref as gref

CODES = (1, 2, 6, 11, 23)
START_SETS = (("ATG",), ("ATG", "GTG", "TTG"), ("ATG", "CTG", "ATA", "ATT"))


def _table(segs):
    from magot_b200.tables import RecordTable
    rec_off = np.concatenate(([0], np.cumsum([len(r) for r in segs])))
    flat = [x for r in segs for x in r]
    cols = [np.array([x[k] for x in flat], dtype=t) for k, t in enumerate((np.int32, np.int64, np.int64, np.int8))]
    n = len(segs)
    names = [b">t%d\n" % i for i in range(n)]
    pre = np.array([len(x) for x in names], dtype=np.int32)
    suf = np.ones(n, dtype=np.int32)
    lit = np.frombuffer(b"".join(x + b"\n" for x in names), dtype=np.uint8)
    lit_off = np.concatenate(([0], np.cumsum(pre.astype(np.int64) + suf)[:-1]))
    return RecordTable(rec_off, *cols, lit_off, pre, suf, lit)


def _orf(S, code=1, starts=("ATG",), min_aa=0, p5=False, p3=False):
    stop, start = ref.code_sets(code, starts)
    return ref.orf_record(S, ref.select(ref.candidates(S, stop, start, p5, p3), min_aa), start)


def _fields(r):
    return (r["lo"], r["hi"], r["n_aa"], r["frame"], ref.ORF_TYPES[r["type"]])


def test_stop_at_the_very_end_and_no_stop():
    r = _orf(b"ATGAAATAA")
    assert _fields(r) == (0, 9, 2, 0, "complete")
    assert r["start_codon"] == cref.codon_index(b"ATG") and r["stop_codon"] == cref.codon_index(b"TAA")
    assert _orf(b"ATGAAAAAAC")["n_aa"] == 0                                   # no stop, no 3' partial
    r = _orf(b"ATGAAAAAAC", p3=True)                                           # through the frame's last complete codon
    assert _fields(r) == (0, 9, 3, 0, "3prime_partial") and r["stop_codon"] == 0xFF
    r = _orf(b"CCATGAAAAAAC", p3=True)
    assert _fields(r) == (2, 11, 3, 2, "3prime_partial")


def test_start_at_a_frames_first_codon_and_5prime_partial():
    assert _fields(_orf(b"ATGAAATAG", p5=True)) == (0, 9, 2, 0, "complete")   # codon f is a start: not partial
    assert _fields(_orf(b"AAAATGTAG")) == (3, 9, 1, 0, "complete")
    r = _orf(b"AAAATGTAG", p5=True)
    assert _fields(r) == (0, 9, 2, 0, "5prime_partial") and r["start_codon"] == cref.codon_index(b"AAA")
    assert _fields(_orf(b"CCCCCC", p5=True, p3=True)) == (0, 6, 2, 0, "internal")
    assert _orf(b"CCATGCC", p5=True, p3=True)["lo"] == 0                        # frame 0 first, two codons; frames 1, 2 shorter
    assert _orf(b"AAATAACCC", p5=True, min_aa=2)["n_aa"] == 0                  # later stretches need a start
    assert _fields(_orf(b"AAATAACCC", p5=True)) == (0, 6, 1, 0, "5prime_partial")


def test_stretch_that_is_only_a_stop():
    S = b"TAAATGCCCTGA"
    assert _fields(_orf(S)) == (3, 12, 2, 0, "complete")
    assert _fields(_orf(S, p5=True)) == (3, 12, 2, 0, "complete")              # the first stretch (a lone stop) has 0 residues
    assert _orf(b"TAA", p5=True)["n_aa"] == 0


def test_min_aa_around_n_aa():
    S = b"ATG" + b"GCC" * 6 + b"TAG"                                           # 7 residues
    for m, n in ((6, 7), (7, 7), (8, 0), (0, 7), (1, 7)):
        assert _orf(S, min_aa=m)["n_aa"] == n


def test_ties_across_frames_take_the_smaller_start():
    S = b"C" + b"ATGAAATAG" + b"C" + b"ATGCCCTGA"                              # frame 1 at 1 and frame 2 at 11, both 2 residues
    assert _fields(_orf(S)) == (1, 10, 2, 1, "complete")
    S = b"CC" + b"ATGAAATAG" + b"ATGCCCTGA"                                    # the same frame, two stretches
    assert _fields(_orf(S)) == (2, 11, 2, 2, "complete")


def test_ambiguous_and_lower_case_codons():
    r = _orf(b"atgNNNtag")
    assert _fields(r) == (0, 9, 2, 0, "complete") and r["start_codon"] == cref.codon_index(b"ATG")
    assert _orf(b"ATGTNATAA")["hi"] == 9                                       # TNA is not a stop
    assert _orf(b"NTGAAATAA")["n_aa"] == 0                                     # NTG is not a start
    r = _orf(b"NTGAAATAA", p5=True)
    assert _fields(r) == (0, 9, 2, 0, "5prime_partial") and r["start_codon"] == 0xFF
    assert _orf(b"ATGAAAtRa", p3=True)["type"] == 2                           # tRa is not a stop


def test_genetic_codes_and_start_sets():
    assert _orf(b"ATGTGAAGA")["n_aa"] == 1                                     # table 1: TGA stops
    assert _fields(_orf(b"ATGTGAAGA", code=2)) == (0, 9, 2, 0, "complete")    # table 2: TGA = W, AGA stops
    assert _orf(b"ATGTAAGCCTGA", code=6)["n_aa"] == 3                          # table 6: TAA = Q
    assert _orf(b"ATGCCCTTA", code=23)["n_aa"] == 2                            # table 23: TTA stops
    assert _orf(b"GTGCCCTAA", code=11)["n_aa"] == 0
    r = _orf(b"GTGCCCTAA", code=11, starts=("ATG", "GTG", "TTG"))
    assert _fields(r) == (0, 9, 2, 0, "complete") and r["start_codon"] == cref.codon_index(b"GTG")


def _walk(S, code, starts, min_aa, p5, p3):
    """The semantics once more, as a plain walk over the codons of each frame."""
    table = gref.table64(code)
    best = None
    n = len(S)
    for f in range(3):
        open_ = f if p5 and f + 3 <= n else None
        last = None
        for i in range(f, n - 2, 3):
            c = cref.codon_index(S[i:i + 3])
            last = i
            if c is not None and table[c] == "*":
                if open_ is not None:
                    cand = ((i - open_) // 3, open_, i + 3, True)
                    if cand[0] >= max(1, min_aa) and (best is None or (cand[0], -cand[1]) > (best[0], -best[1])):
                        best = cand
                open_ = None
            elif open_ is None and c is not None and S[i:i + 3].upper().decode() in starts:
                open_ = i
        if p3 and open_ is not None:
            cand = ((last + 3 - open_) // 3, open_, last + 3, False)
            if cand[0] >= max(1, min_aa) and (best is None or (cand[0], -cand[1]) > (best[0], -best[1])):
                best = cand
    return best


def test_model_against_a_codon_walk():
    rng = np.random.default_rng(1)
    alpha = np.frombuffer(b"ACGTACGTACGTacgtNRTAATGA", dtype=np.uint8)
    payloads = [alpha[rng.integers(0, alpha.size, size=int(n))].tobytes() for n in rng.integers(0, 400, size=60)]
    payloads += [b"", b"A", b"AT", b"ATG", b"TAA"]
    for code in CODES:
        for starts in START_SETS:
            stop, start = ref.code_sets(code, starts)
            if any(stop[cref.codon_index(c.encode())] for c in starts):
                continue
            for p5 in (False, True):
                for p3 in (False, True):
                    for S in payloads:
                        cands = ref.candidates(S, stop, start, p5, p3)
                        for m in (0, 1, 30, 100):
                            assert ref.select(cands, m) == _walk(S, code, starts, m, p5, p3), (code, starts, p5, p3, S, m)


def test_mapping_and_phases_plus_and_minus():
    rng = np.random.default_rng(4)
    contig = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=3000).tobytes()
    recs = [
        [(0, 101, 130, 0), (0, 201, 240, 0), (0, 301, 335, 0)],
        [(0, 301, 335, 1), (0, 201, 240, 1), (0, 101, 130, 1)],
        [(0, 5000, 5100, 0), (0, 11, 30, 0), (0, 50, 49, 0), (0, -40, -1, 0), (0, 61, 99, 0)],   # clamped away, empty, negative
        [(0, 61, 99, 1), (0, -40, -1, 1), (0, 50, 49, 1), (3, 1, 10, 1), (0, 11, 30, 1)],      # a contig outside the genome
    ]
    tbl = _table(recs)
    for r in range(tbl.n_rec):
        S = cref.payload([contig], tbl, r)
        segs = ref.clamped_segments([contig], tbl, r)
        for lo, hi in ((0, len(S)), (1, len(S) - 2), (31, 32), (len(S) - 3, len(S))):
            m = ref.map_segments(segs, lo, hi)
            parts, done = [], 0
            for (a, b, ph), (cl, ch, minus) in zip(m, segs):
                if a < 0:
                    assert (a, b, ph) == (-1, -1, -1)
                    continue
                assert cl <= a < b <= ch
                assert ph == (3 - done % 3) % 3                                # bases of the ORF before the segment
                s = contig[a:b]
                parts.append(gref.revcomp(s) if minus else s)
                done += b - a
            assert b"".join(parts) == S[lo:hi]
    # a clamped-away segment is never touched, and the phases of a 3-segment ORF
    m = ref.map_segments(ref.clamped_segments([contig], tbl, 0), 10, 80)
    assert [x[2] for x in m] == [0, 1, 0] and m[0] == (110, 130, 0)
    m = ref.map_segments(ref.clamped_segments([contig], tbl, 1), 10, 80)
    assert m[0] == (300, 325, 0) and m[1][2] == 2


def test_antisense_table():
    from magot_b200 import genome
    rng = np.random.default_rng(5)
    contig = rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), size=2000).tobytes()
    recs = [[(0, 11, 30, 0), (0, 51, 90, 0)], [(0, 51, 90, 1), (0, 11, 30, 1)], [], [(0, 5, 4, 0), (0, -30, -1, 1), (0, 400, 450, 0)]]
    tbl = _table(recs)
    cols = ref.antisense(tbl)
    at = genome.antisense_table(tbl)
    for a, b in zip(cols, (at.rec_seg_off, at.seg_contig, at.seg_start, at.seg_end, at.seg_strand)):
        assert np.array_equal(a, b)
    assert np.array_equal(at.lit, tbl.lit) and np.array_equal(at.rec_pre_len, tbl.rec_pre_len)
    for r in range(tbl.n_rec):
        assert cref.payload([contig], at, r) == gref.revcomp(cref.payload([contig], tbl, r))


def _prediction(contigs, tbl, **kw):
    """A genome.CdsPrediction built from the model's results (sense only)."""
    from magot_b200 import engine, genome
    recs, segs = ref.predict(contigs, tbl, **kw)
    rec = np.zeros(len(recs), dtype=engine.PRED_DTYPE)
    for i, r in enumerate(recs):
        for f in ref.FIELDS:
            rec[f][i] = r[f]
    seg = np.array(segs, dtype=np.int64).reshape(-1, 3)
    keep = seg[:, 0] >= 0
    return genome.CdsPrediction(["t%d" % i for i in range(len(recs))], rec, np.zeros(len(recs), np.int8),
                                tbl.seg_contig[keep], seg[keep, 0], seg[keep, 1], tbl.seg_strand[keep], seg[keep, 2].astype(np.int8),
                                np.concatenate(([0], np.cumsum(rec["n_cds_seg"]))))


def test_three_text_formats():
    from magot_b200 import genome_tools
    #          exon 1 (ATG..)     intron   exon 2 (..TAA)
    contig = b"CCATGAAACC" + b"GTAAAG" + b"CGGGTTTTAACC" + b"A" * 30
    recs = [[(0, 3, 10, 0), (0, 17, 28, 0)], [(0, 31, 40, 0)],                 # a spliced ORF; a record without an ORF
            [(0, 17, 28, 1), (0, 3, 10, 1)]]                                   # the same exons on '-'
    tbl = _table(recs)
    pred = _prediction([contig], tbl, min_aa=1)
    assert list(pred.records["n_aa"]) == [5, 0, pred.records["n_aa"][2]]
    lines = genome_tools._predict_lines(pred, {0: "chr1"}, "gff3")
    assert lines[0] == "##gff-version 3"
    assert lines[1:3] == ["chr1\tmagot_b200\tCDS\t3\t10\t.\t+\t0\tID=t0.cds;Parent=t0;orf_type=complete;length_aa=5",
                          "chr1\tmagot_b200\tCDS\t17\t26\t.\t+\t1\tID=t0.cds;Parent=t0;orf_type=complete;length_aa=5"]
    assert all("Parent=t1" not in x for x in lines)
    t2 = [x.split("\t") for x in lines if "Parent=t2;" in x]
    assert [int(x[3]) for x in t2] == sorted(int(x[3]) for x in t2) and all(x[6] == "-" for x in t2)
    has = np.flatnonzero(pred.records["n_aa"] > 0)
    S = [cref.payload([contig], tbl, int(r)) for r in has]
    cds = [s[int(pred.records["lo"][r]):int(pred.records["hi"][r])].decode() for s, r in zip(S, has)]
    assert cds[0] == "ATGAAACC" + "CGGGTTTTAA"
    lines = genome_tools._predict_lines(pred, {0: "chr1"}, "cds", cds)
    assert lines[0] == ">t0.p1 orf_type=complete len=5 t0:1-18(+)" and lines[1] == cds[0]
    prot = [gref.translate(c.encode(), gref.table64(1), trimX=False).decode() for c in cds]
    lines = genome_tools._predict_lines(pred, {0: "chr1"}, "protein", prot)
    assert lines[1] == "MKPGF*" and len(lines) == 2 * has.size


def test_tool_argument_errors(tmp_path):
    from magot_b200 import genome_tools
    missing = str(tmp_path / "missing")
    with pytest.raises(ValueError, match="genetic_code"):
        genome_tools.predict_cds(missing, missing, genetic_code="7")
    with pytest.raises(ValueError, match="out_format"):
        genome_tools.predict_cds(missing, missing, out_format="gtf")
    with pytest.raises(ValueError, match="partial"):
        genome_tools.predict_cds(missing, missing, partial="True")
    with pytest.raises(ValueError, match="strand"):
        genome_tools.predict_cds(missing, missing, strand="minus")
    with pytest.raises(ValueError, match="min_orf"):
        genome_tools.predict_cds(missing, missing, min_orf="-1")
    with pytest.raises(ValueError, match="min_orf"):
        genome_tools.predict_cds(missing, missing, min_orf="ten")
    with pytest.raises(ValueError, match="stop codon"):
        genome_tools.predict_cds(missing, missing, start_codons="ATG,TAG")
    with pytest.raises(ValueError, match="A/C/G/T"):
        genome_tools.predict_cds(missing, missing, start_codons="AUG")
    with pytest.raises(ValueError, match="strand"):
        genome_tools.main(["genome_tools", "predict_cds", missing, missing, "strand=antisense"])
