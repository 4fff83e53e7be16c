"""CDS prediction on the device (mg_plan_predict_cds*, engine.Plan.predict_cds, AnnotationSet.predict_cds, genome_tools
predict_cds), bit for bit against the numpy model cdspredict_ref: random genomes over the full alphabet and random tables (empty,
clamped-away and negative segments, 1-2 base records, a record of several 32 KB tiles, thousands of tiny segments in one tile, a
stop-free record of several warp steps), five genetic codes, three start sets, the four partial combinations, min_aa 0, 1, 30 and
100, both strands; three kinds of prepare under both K1 variants; NULL seg_out; the state checks; CUDA graphs; the ORF against
the nucleotide text; the O. biroi RefSeq fixture with a check_cds round trip; a genome past forward index 2^31 and reverse-plane
index 2^32 with segments of 2^31 bases or more."""
import contextlib
import ctypes
import gzip
import io
import os

import numpy as np
import pytest

import cdscheck_ref as cref
import cdspredict_ref as ref
import gencode_ref as gref
from test_gpu_check import CODES, START_SETS, _genome, _random_case, _starts, _table

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
PARTIALS = ((False, False), (True, False), (False, True), (True, True))
MIN_AA = (0, 1, 30, 100)


@pytest.fixture(scope="module")
def mg():
    import magot_b200
    return magot_b200


@pytest.fixture()
def k1_mode(mg):
    from magot_b200 import _lib
    yield lambda v: _lib.check(_lib.lib.mg_tune(b"k1", v))
    _lib.check(_lib.lib.mg_tune(b"k1", 0))


def _case(rng, n_rec=400):
    """_random_case plus a contig of A/C only (no stop and no start in any of the five codes) and a 5 000-base record on it:
    stop-free over ten warp steps."""
    contigs, segs, _ = _random_case(rng, n_rec)
    contigs.append(np.frombuffer(b"ACac", dtype=np.uint8)[rng.integers(0, 4, size=6000)].tobytes())
    segs.append([(len(contigs) - 1, 3, 5002, 0)])
    segs.append([(len(contigs) - 1, 1, 4000, 1)])
    return contigs, segs


def _check(got, want):
    msg = ref.compare(got[0], got[1], want[0], want[1])
    assert msg is None, msg


@pytest.mark.parametrize("code", CODES)
def test_random_tables_codes_starts_partials(mg, code):
    from magot_b200 import engine, gencode, genome
    rng = np.random.default_rng(0)
    contigs, segs = _case(rng)
    tbl = _table(segs)
    tables = [tbl] + ([genome.antisense_table(tbl)] if code in (1, 2) else [])
    g = _genome(contigs)
    try:
        for t in tables:
            plan = engine.Plan(g, t)
            if code != 1:
                plan.set_codon_table(gencode.codon64(code))
            plan.prepare(trimx=False)
            cache = {}
            for which in START_SETS:
                starts = _starts(code, which)
                for p5, p3 in PARTIALS:
                    for m in MIN_AA:
                        want = ref.predict(contigs, t, code, starts, m, p5, p3, cache)
                        _check(plan.predict_cds(m, gencode.start64(starts, code), p5, p3), want)
            plan.close()
    finally:
        g.close()


@pytest.mark.parametrize("k1", [0, 1])
@pytest.mark.parametrize("prep", ["sync", "async", "defer"])
def test_prepare_kinds_and_null_seg_out(mg, k1_mode, k1, prep):
    import torch
    from magot_b200 import engine, _lib
    k1_mode(k1)
    rng = np.random.default_rng(7)
    contigs, segs = _case(rng, 200)
    tbl = _table(segs, framing=(prep != "defer"))
    want = ref.predict(contigs, tbl, 1, ("ATG",), 30, True, True)
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        if prep == "sync":
            plan.prepare()
        else:
            plan.prepare_async(defer_records=(prep == "defer"))
        _check(plan.predict_cds(30, None, True, True), want)
        flags = _lib.MG_PRED_5PARTIAL | _lib.MG_PRED_3PARTIAL
        recs = np.zeros(tbl.n_rec, dtype=engine.PRED_DTYPE)
        _lib.check(_lib.lib.mg_plan_predict_cds(plan.handle, 30, None, flags, ctypes.c_void_p(recs.ctypes.data), None, None))
        _lib.check(_lib.lib.mg_stream_sync(0, None))
        _check((recs, None), want)
        for with_seg in (False, True):                   # the device variant into poisoned buffers
            d_rec = torch.full((tbl.n_rec * 32,), 0xA5, dtype=torch.uint8, device="cuda")
            d_seg = torch.full((tbl.n_seg * 24,), 0x5A, dtype=torch.uint8, device="cuda") if with_seg else None
            _lib.check(_lib.lib.mg_plan_predict_cds_device(plan.handle, 30, None, flags, ctypes.c_void_p(d_rec.data_ptr()),
                                                           ctypes.c_void_p(d_seg.data_ptr()) if with_seg else None, None))
            torch.cuda.synchronize()
            got_seg = d_seg.cpu().numpy().view(engine.CDSSEG_DTYPE) if with_seg else None
            _check((d_rec.cpu().numpy().view(engine.PRED_DTYPE), got_seg), want)
        plan.close()
    finally:
        g.close()


def test_orf_against_nucleotide_text(mg):
    """The reported ORF is S[lo:hi] of the record's K2 text: its first codon is start_codon, its last stop_codon, and it has no
    other in-frame stop."""
    from magot_b200 import engine, gencode
    rng = np.random.default_rng(3)
    contigs, segs = _case(rng, 300)
    tbl = _table(segs, framing=False)
    g = _genome(contigs)
    try:
        for code in (1, 2):
            plan = engine.Plan(g, tbl)
            if code != 1:
                plan.set_codon_table(gencode.codon64(code))
            plan.prepare(trimx=False)
            recs, _ = plan.predict_cds(1, gencode.start64(("ATG", "GTG"), code), True, True)
            text = plan.emit_bytes()
            nuc, _ = plan.lengths()
            off = np.concatenate(([0], np.cumsum(nuc)))
            stop, _ = ref.code_sets(code, ("ATG",))
            n_orf = 0
            for r in range(tbl.n_rec):
                S = text[off[r]:off[r + 1]]
                assert S == cref.payload(contigs, tbl, r)
                lo, hi = int(recs["lo"][r]), int(recs["hi"][r])
                if lo < 0:
                    continue
                n_orf += 1
                orf = S[lo:hi]
                idx = [cref.codon_index(orf[i:i + 3]) for i in range(0, len(orf), 3)]
                assert (idx[0] if idx[0] is not None else 0xFF) == int(recs["start_codon"][r])
                has_stop = not int(recs["type"][r]) & 2
                assert (idx[-1] if has_stop else 0xFF) == int(recs["stop_codon"][r])
                inner = idx[:-1] if has_stop else idx
                assert not any(c is not None and stop[c] for c in inner) and len(inner) == int(recs["n_aa"][r])
            assert n_orf > 100
            plan.close()
    finally:
        g.close()


def test_argument_and_state_errors(mg):
    from magot_b200 import engine, gencode, _lib
    contigs = [b"ATGAAATAG" * 100]
    tbl = _table([[(0, 1, 9, 0)]])
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        recs = np.zeros(1, dtype=engine.PRED_DTYPE)
        P = ctypes.c_void_p(recs.ctypes.data)
        assert _lib.lib.mg_plan_predict_cds(plan.handle, 0, None, 0, P, None, None) == -4          # not prepared
        plan.prepare_async(defer_records=True)
        assert _lib.lib.mg_plan_predict_cds(plan.handle, 0, None, 4, P, None, None) == -1
        assert _lib.lib.mg_plan_predict_cds(plan.handle, 0, bytes(64), 0, P, None, None) == -1
        assert "no start codon" in _lib.last_error()
        assert _lib.lib.mg_plan_predict_cds(plan.handle, 0, gencode.start64(["TAA"], 6), 0, P, None, None) == -1
        assert "stop codon" in _lib.last_error()
        assert _lib.lib.mg_plan_predict_cds(plan.handle, 0, None, 0, None, None, None) == -1
        r, s = plan.predict_cds(0)
        assert (int(r["lo"][0]), int(r["hi"][0]), int(r["n_aa"][0]), int(r["n_cds_seg"][0])) == (0, 9, 2, 1)
        assert (int(s["lo"][0]), int(s["hi"][0]), int(s["phase"][0])) == (0, 9, 0)
        assert plan.predict_cds(3)[0]["n_aa"][0] == 0 and plan.predict_cds(1 << 40)[0]["n_aa"][0] == 0
        g.mask([0], [3], [6], hard=True)
        assert _lib.lib.mg_plan_predict_cds(plan.handle, 0, None, 0, P, None, None) == -4          # genome changed
        assert "prepare it again" in _lib.last_error()
        assert _lib.lib.mg_plan_predict_cds_device(plan.handle, 0, None, 0, P, None, None) == -4
        plan.close()
    finally:
        g.close()


def test_graph_capture_and_replay(mg):
    import torch
    from magot_b200 import engine, _lib
    L = _lib.lib
    rng = np.random.default_rng(5)
    contigs, segs = _case(rng, 300)
    tbl = _table(segs)
    want = ref.predict(contigs, tbl, 1, ("ATG",), 30, False, True)
    g = _genome(contigs)
    s = torch.cuda.Stream()
    sp = ctypes.c_void_p(s.cuda_stream)
    try:
        plan = engine.Plan(g, tbl, stream=sp)
        plan.prepare_async()
        n, e = tbl.n_rec, tbl.n_seg
        d_rec = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
        d_seg = torch.empty(e * 24, dtype=torch.uint8, device="cuda")
        cap_n, cap_p = plan.capacities()
        torch.cuda.synchronize()
        _lib.check(L.mg_graph_begin(0, sp))
        try:
            _lib.check(L.mg_plan_prepare_async(plan.handle, _lib.MG_PROT_DEFER, cap_n, cap_p, sp))
            _lib.check(L.mg_plan_predict_cds_device(plan.handle, 30, None, _lib.MG_PRED_3PARTIAL, ctypes.c_void_p(d_rec.data_ptr()),
                                                    ctypes.c_void_p(d_seg.data_ptr()), sp))
        finally:
            gx = ctypes.c_void_p()
            _lib.check(L.mg_graph_end(0, sp, ctypes.byref(gx)))
        for _ in range(3):
            d_rec.fill_(0xA5)
            d_seg.fill_(0x5A)
            torch.cuda.synchronize()
            _lib.check(L.mg_graph_launch(0, gx, sp))
            s.synchronize()
            _check((d_rec.cpu().numpy().view(engine.PRED_DTYPE), d_seg.cpu().numpy().view(engine.CDSSEG_DTYPE)), want)
        _lib.check(L.mg_graph_destroy(gx))
        # the host variant allocates its device outputs on first use: inside a capture that is refused, outside it works
        plan2 = engine.Plan(g, tbl, stream=sp)
        plan2.prepare()
        recs = np.zeros(n, dtype=engine.PRED_DTYPE)
        torch.cuda.synchronize()
        _lib.check(L.mg_graph_begin(0, sp))
        rc = L.mg_plan_predict_cds(plan2.handle, 30, None, 0, ctypes.c_void_p(recs.ctypes.data), None, sp)
        err = _lib.last_error()
        gx = ctypes.c_void_p()
        _lib.check(L.mg_graph_end(0, sp, ctypes.byref(gx)))
        _lib.check(L.mg_graph_destroy(gx))
        assert rc == -4 and "capture" in err
        _check(plan2.predict_cds(30, None, False, True), want)
        plan.close()
        plan2.close()
    finally:
        g.close()


def _stdout_of(fn, *a, **k):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        fn(*a, **k)
    return buf.getvalue()


def test_obiroi_predict_and_check_round_trip(mg, tmp_path):
    """The exon models of the O. biroi RefSeq fixture: the prediction against the model, the number of mRNAs whose predicted CDS
    is the annotated one, and a round trip: the GFF without its CDS rows plus the predicted rows, read back and checked."""
    from magot_b200 import genome, genome_tools
    from magot_b200.genome import _native_table, _PENDING
    d = os.path.join(HERE, "golden", "ref_test_data")
    fa, gff = tmp_path / "g.fa", tmp_path / "a.gff"
    fa.write_bytes(gzip.open(os.path.join(d, "O.biroi_refseqGenomeSubset.fasta.gz")).read())
    gff.write_bytes(gzip.open(os.path.join(d, "O.biroi_NCBIrefseq_gff3Subset.gff.gz")).read())
    g = genome.Genome(str(fa))
    g.read_gff(str(gff), base_features=["exon"], features_to_ignore=["CDS"])
    gs, tbl, _ = _native_table(g.annotations, _PENDING.get(g.annotations), "gene")
    names = list(gs)
    contigs = [None] * len(names)
    for n in names:
        contigs[gs.contig_index(n)] = str(gs[n]).encode("latin-1")
    pred = g.annotations.predict_cds("gene", min_aa=100)
    keep = np.flatnonzero(tbl.rec_pre_len > 0)
    recs, segs = ref.predict(contigs, tbl, min_aa=100)
    assert ref.compare(pred.records, None, [recs[r] for r in keep], None) is None
    want_segs = [s for r in keep.tolist() for s in segs[tbl.rec_seg_off[r]:tbl.rec_seg_off[r + 1]] if s[0] >= 0]
    assert [(int(a), int(b), int(p)) for a, b, p in zip(pred.seg_lo, pred.seg_hi, pred.seg_phase)] == want_segs
    # the object model (the set materialised) gives the same result
    g2 = genome.Genome(str(fa))
    g2.read_gff(str(gff), base_features=["exon"], features_to_ignore=["CDS"])
    assert len(g2.annotations.gene) > 0
    obj = g2.annotations.predict_cds("gene", min_aa=100)
    assert obj.names == pred.names and ref.compare(obj.records, None, [recs[r] for r in keep], None) is None
    # mRNAs whose predicted CDS is the annotated one, segment for segment
    g3 = genome.Genome(str(fa))
    g3.read_gff(str(gff))
    cs, ctbl, _ = _native_table(g3.annotations, _PENDING.get(g3.annotations), "gene")
    ckeep = np.flatnonzero(ctbl.rec_pre_len > 0)
    annotated = {}
    for n, r in zip(genome._record_names(ctbl, ckeep), ckeep.tolist()):
        annotated[n] = sorted(cref.clamp(len(contigs[ctbl.seg_contig[e]]), ctbl.seg_start[e], ctbl.seg_end[e])
                              for e in range(ctbl.rec_seg_off[r], ctbl.rec_seg_off[r + 1]))
    agree = 0
    for i, n in enumerate(pred.names):
        got = sorted(zip(pred.seg_lo[pred.seg_off[i]:pred.seg_off[i + 1]].tolist(), pred.seg_hi[pred.seg_off[i]:pred.seg_off[i + 1]].tolist()))
        agree += n in annotated and got == annotated[n]
    print("O. biroi predict_cds: %d of %d mRNAs agree with the annotated CDS (%d transcripts)" % (agree, len(annotated), len(pred.names)))
    assert (agree, len(annotated), len(pred.names)) == OBIROI_AGREE
    # round trip through check_cds
    out = _stdout_of(genome_tools.main, ["genome_tools", "predict_cds", str(fa), str(gff)])
    rows = out.split("\n")
    assert rows[0] == "##gff-version 3" and rows[-1] == ""
    assert rows[1:-1] == genome_tools._predict_lines(pred, {gs.contig_index(n): n for n in gs}, "gff3")[1:]
    kept = [line for line in gff.read_text(encoding="latin-1").split("\n") if line.count("\t") < 8 or line.split("\t")[2] != "CDS"]
    rt = tmp_path / "rt.gff"
    rt.write_text("\n".join(kept).rstrip("\n") + "\n" + "\n".join(rows[1:]), encoding="latin-1")
    g4 = genome.Genome(str(fa))
    g4.read_gff(str(rt))
    chk = g4.annotations.check_cds("gene")
    status = dict(zip(chk.names, chk.records["flags"].tolist()))
    allowed = 16 | 32                                   # NONCANONICAL_SPLICE (the exons), AMBIGUOUS (an N inside an ORF)
    for i, n in enumerate(pred.names):
        if int(pred.records["n_aa"][i]) > 0 and int(pred.records["type"][i]) == 0:
            assert status[n] & ~allowed == 0, (n, status[n])
    g5 = genome.Genome(str(fa))
    g5.read_gff(str(rt))
    text = g5.annotations.get_fasta("gene", seq_type="protein")
    lines = text.split("\n")
    got = {lines[k][1:]: lines[k + 1] for k in range(len(lines) - 1) if lines[k].startswith(">")}
    prot = _stdout_of(genome_tools.main, ["genome_tools", "predict_cds", str(fa), str(gff), "out_format=protein"]).split("\n")
    for head, seq in zip(prot[0:-1:2], prot[1::2]):
        tid = head[1:].split(".p1 ")[0]
        assert got[tid][1:] == seq[1:] and seq[0] == "M" and got[tid][0] in "MVL", tid
    cds = _stdout_of(genome_tools.main, ["genome_tools", "predict_cds", str(fa), str(gff), "out_format=cds"]).split("\n")
    assert [h for h in cds[0:-1:2]] == [h for h in prot[0:-1:2]]
    for head, seq in zip(cds[0:-1:2], cds[1::2]):
        i = pred.names.index(head[1:].split(".p1 ")[0])
        r = keep[i]
        assert seq.encode() == cref.payload(contigs, tbl, r)[int(pred.records["lo"][i]):int(pred.records["hi"][i])]


#: (mRNAs whose predicted CDS equals the annotated one, annotated mRNAs, exon-model transcripts) on the O. biroi RefSeq subset,
#: min_orf 100, table 1, ATG, sense, no partials
OBIROI_AGREE = (85, 85, 93)


def test_strand_both(mg):
    """strand="both": per record the longer of the sense and the antisense ORF, the sense one on a tie, with the antisense
    table's segments (reversed, strands flipped)."""
    from magot_b200 import engine, genome
    rng = np.random.default_rng(9)
    contigs, segs = _case(rng, 300)
    tbl = _table(segs)
    g = _genome(contigs)
    try:
        sense = engine.Plan(g, tbl)
        sense.prepare()
        at = genome.antisense_table(tbl)
        anti = engine.Plan(g, at)
        anti.prepare()
        rs, ss = sense.predict_cds(30)
        ra, sa = anti.predict_cds(30)
        cols = ref.antisense(tbl)
        assert all(np.array_equal(a, b) for a, b in zip(cols, (at.rec_seg_off, at.seg_contig, at.seg_start, at.seg_end, at.seg_strand)))
        _check((ra, sa), ref.predict(contigs, at, min_aa=30))
        assert (ra["n_aa"] > rs["n_aa"]).any() and (ra["n_aa"] < rs["n_aa"]).any()
        sense.close()
        anti.close()
    finally:
        g.close()


def test_large_genome_past_2e31(mg):
    """Records on a contig that starts past forward index 2^31, '-' records whose reverse-plane indices lie past 2^32, and
    segments of 2^31 bases or more, which the plan splits into chunks: results stay per caller segment."""
    import torch
    from magot_b200 import engine
    big = (1 << 31) + 4096
    need_dev, need_host = big + (1 << 28), 2 * big
    free_dev = torch.cuda.mem_get_info()[0]
    try:
        free_host = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    except (ValueError, OSError):
        free_host = need_host
    if free_dev < need_dev or free_host < need_host:
        pytest.skip("needs %d B of free device memory (%d free) and %d B of free host memory (%d free)"
                    % (need_dev, free_dev, need_host, free_host))
    rng = np.random.default_rng(17)
    block = np.frombuffer(b"ACGTACGTacgtNRGTAG", dtype=np.uint8)[rng.integers(0, 18, size=1 << 20)]
    filler = np.tile(block, big // block.size + 1)[:big]
    alpha = np.frombuffer(b"ACGTACGTACGTacgtN-GTAGGCAGATAC", dtype=np.uint8)
    small = [alpha[rng.integers(0, 30, size=300000)].tobytes() for _ in range(2)]
    g = engine.DeviceGenome([len(small[0]), big, len(small[1])], device=0)
    try:
        g.pack(0, np.frombuffer(small[0], dtype=np.uint8))
        g.pack(1, filler)
        g.pack(2, np.frombuffer(small[1], dtype=np.uint8))
        g.finalize()
        contigs = [small[0], filler.tobytes(), small[1]]
        segs = []
        for r in range(400):
            c = 2 if r % 2 else 0
            m = (r // 2) % 2
            pos = int(rng.integers(1, 290000))
            row = []
            for _ in range(int(rng.integers(1, 6))):
                ln = int(rng.integers(1, 300))
                row.append((c, pos, min(pos + ln - 1, 299999), m))
                pos += ln + int(rng.integers(0, 40))
            segs.append(row[::-1] if m else row)
        segs.append([(1, big - 5000, big, 1), (2, 1, 3000, 1)])
        segs.append([(1, 100, 3000, 0), (1, 3100, 9000, 0)])
        tbl = _table(segs)
        plan = engine.Plan(g, tbl)
        plan.prepare()
        for p5, p3 in PARTIALS:
            _check(plan.predict_cds(1, None, p5, p3), ref.predict(contigs, tbl, min_aa=1, partial5=p5, partial3=p3))
        plan.close()
        # segments of 2^31 bases or more, which the plan splits into chunks: the mapping is per caller segment, and the ORF's
        # first and last codons, read from the genome at the mapped coordinates, are the reported ones
        long_segs = [[(1, 1, big - 100, 0), (1, big - 90, big - 10, 0)], [(1, big - 90, big - 10, 1), (1, 1, big - 100, 1)],
                     [(0, 1, 500, 0), (1, 1, big, 0), (1, 20, 80, 0)], [(1, -big, -1, 1), (2, 1, 10, 1)]]
        tbl = _table(long_segs)
        plan = engine.Plan(g, tbl)
        plan.prepare_async(defer_records=True)
        recs, sg = plan.predict_cds(1, None, True, True)
        plan.close()
        for r in range(tbl.n_rec):
            assert int(recs["n_aa"][r]) > 0
            e0, e1 = int(tbl.rec_seg_off[r]), int(tbl.rec_seg_off[r + 1])
            clamped = ref.clamped_segments(contigs, tbl, r)
            m = ref.map_segments(clamped, int(recs["lo"][r]), int(recs["hi"][r]))
            assert [(int(a), int(b), int(p)) for a, b, p in zip(sg["lo"][e0:e1], sg["hi"][e0:e1], sg["phase"][e0:e1])] == m
            assert int(recs["n_cds_seg"][r]) == sum(1 for x in m if x[0] >= 0)
            parts = [(contigs[int(tbl.seg_contig[e])], x, minus) for e, x, (_, _, minus) in zip(range(e0, e1), m, clamped) if x[0] >= 0]
            first, last = parts[0], parts[-1]
            head = first[0][first[1][1] - 3:first[1][1]] if first[2] else first[0][first[1][0]:first[1][0] + 3]
            tail = last[0][last[1][0]:last[1][0] + 3] if last[2] else last[0][last[1][1] - 3:last[1][1]]
            head, tail = (gref.revcomp(head) if first[2] else head), (gref.revcomp(tail) if last[2] else tail)
            sc = cref.codon_index(head)
            assert (0xFF if sc is None else sc) == int(recs["start_codon"][r])
            if not int(recs["type"][r]) & 2:
                assert cref.codon_index(tail) == int(recs["stop_codon"][r])
    finally:
        g.close()
