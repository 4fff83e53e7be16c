"""The gene-model check on the device (mg_plan_check*, engine.Plan.check, AnnotationSet.check_cds, genome_tools check_cds),
bit for bit against the numpy model cdscheck_ref: random genomes over the full alphabet, random tables (empty, clamped-away and
negative segments, 1-2 base records, codons across segment and tile boundaries, a record of several tiles, thousands of tiny
segments in one tile), five genetic codes, three start sets, with and without the phase; three kinds of prepare under both K1
variants; every NULL combination of the optional outputs; agreement with the protein text; masks; CUDA graphs; the O. biroi
RefSeq fixture; a genome past forward index 2^31 and reverse-plane index 2^32."""
import contextlib
import ctypes
import gzip
import io
import os

import numpy as np
import pytest

import cdscheck_ref as ref
import gencode_ref as gref

pytestmark = pytest.mark.gpu

CODES = (1, 2, 6, 11, 23)
SENSE = tuple("ACGT"[i >> 4] + "ACGT"[(i >> 2) & 3] + "ACGT"[i & 3] for i in range(64))
START_SETS = (("ATG",), ("ATG", "GTG", "TTG"), "sense")
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def mg():
    import magot_b200
    return magot_b200


@pytest.fixture()
def k1_mode(mg):
    from magot_b200 import _lib
    yield lambda v: _lib.check(_lib.lib.mg_tune(b"k1", v))
    _lib.check(_lib.lib.mg_tune(b"k1", 0))


def _starts(code, which):
    if which != "sense":
        return which
    t = gref.table64(code)
    return tuple(c for c in SENSE if t["ACGT".index(c[0]) * 16 + "ACGT".index(c[1]) * 4 + "ACGT".index(c[2])] != "*")


def _genome(contigs):
    from magot_b200 import engine
    g = engine.DeviceGenome([len(c) for c in contigs], device=0)
    for i, c in enumerate(contigs):
        g.pack(i, np.frombuffer(c, dtype=np.uint8))
    g.finalize()
    return g


def _table(segs, phase=None, framing=True):
    from magot_b200 import engine
    rec_off = np.concatenate(([0], np.cumsum([len(r) for r in segs]))).astype(np.int64)
    flat = [x for r in segs for x in r]
    cols = [np.array([x[k] for x in flat], dtype=t) for k, t in enumerate((np.int32, np.int64, np.int64, np.int8))]
    n = len(segs)
    names = [b">r%d\n" % i for i in range(n)] if framing else [b""] * n
    pre = np.array([len(x) for x in names], dtype=np.int32)
    suf = np.full(n, 1 if framing else 0, dtype=np.int32)
    lit = np.frombuffer(b"".join(x + (b"\n" if framing else b"") for x in names), dtype=np.uint8)
    lit_off = np.concatenate(([0], np.cumsum(pre.astype(np.int64) + suf)[:-1])) if n else np.zeros(0, np.int64)
    return engine.RecordTable(rec_off, *cols, lit_off, pre, suf, lit, None if phase is None else np.asarray(phase, np.int8))


def _random_case(rng, n_rec=400):
    alpha = np.frombuffer(b"ACGTACGTACGTACGTacgtacgtNnRYKM-*xSGTAGGCAGATAC", dtype=np.uint8)
    contigs = []
    for n in (0, 3, 1000, 40000, 70000, 150000):
        a = alpha[rng.integers(0, alpha.size, size=n)].copy()
        for _ in range(n // 5000):                          # N runs and lower-case runs
            k = int(rng.integers(0, max(1, n - 300)))
            run = a[k:k + int(rng.integers(1, 300))]
            run[:] = ord("N") if rng.integers(0, 2) else np.frombuffer(run.tobytes().lower(), dtype=np.uint8)
        contigs.append(a.tobytes())
    L = np.array([len(c) for c in contigs], dtype=np.int64)
    segs = []
    for r in range(n_rec):
        kind = r % 10
        if kind == 0:
            segs.append([])
            continue
        c = int(rng.integers(2, len(contigs)))
        m = bool(rng.integers(0, 2))
        if kind == 1:                                       # 1-2 base record
            a = int(rng.integers(1, L[c] - 3))
            segs.append([(c, a, a + int(rng.integers(0, 2)), int(m))])
            continue
        k = int(rng.integers(1, 9))
        pos = int(rng.integers(1, max(2, L[c] - 4000)))
        row = []
        for _ in range(k):                                  # an exon chain with introns of 0..60 bases, sometimes shuffled
            ln = int(rng.integers(1, 400))
            row.append((c, pos, pos + ln - 1, int(m)))
            pos += ln + int(rng.integers(0, 60))
        if m:
            row.reverse()
        if kind == 2 and len(row) > 1:
            row[0], row[1] = row[1], row[0]
        if kind == 3:                                       # negative and clamped-away segments, a contig change
            row.append((c, -int(rng.integers(1, 500)), -int(rng.integers(0, 2)), int(m)))
            row.append((c, L[c] + 5, L[c] + 50, int(m)))
            row.append((0, 1, 10, int(m)))
            row.append((int(rng.integers(1, len(contigs))), 5, 300, int(not m)))
        segs.append(row)
    segs.append([(5, 1, 140000, 0)])                        # one record of several 32 KB tiles
    segs.append([(5, 1 + 7 * k, 4 + 7 * k, 1) for k in range(6000)][::-1])   # thousands of 4-base segments in one tile
    phase = rng.integers(-1, 4, size=len(segs))
    return contigs, segs, phase


def _assert_same(got, want, contigs, tbl):
    recs, counts, junc = got
    w_recs, w_counts, w_junc = want
    msg = ref.compare(recs, w_recs)
    assert msg is None, msg
    if counts is not None:
        assert np.array_equal(counts.astype(np.int64), w_counts)
    if junc is not None:
        assert np.array_equal(junc, w_junc)


@pytest.mark.parametrize("seed", [0, 1])
def test_random_tables_codes_starts_phase(mg, seed):
    from magot_b200 import engine, gencode
    rng = np.random.default_rng(seed)
    contigs, segs, phase = _random_case(rng)
    tbl = _table(segs, phase)
    g = _genome(contigs)
    try:
        for code in CODES:
            plan = engine.Plan(g, tbl)
            if code != 1:
                plan.set_codon_table(gencode.codon64(code))
            plan.prepare(trimx=False)
            for which in START_SETS:
                starts = _starts(code, which)
                for use_phase in (False, True):
                    want = ref.check(contigs, tbl, code, starts, use_phase)
                    _assert_same(plan.check(gencode.start64(starts, code), use_phase, True, True), want, contigs, tbl)
            plan.close()
    finally:
        g.close()


@pytest.mark.parametrize("k1", [0, 1])
@pytest.mark.parametrize("prep", ["sync", "async", "defer"])
def test_prepare_kinds_and_null_outputs(mg, k1_mode, k1, prep):
    from magot_b200 import engine, _lib
    k1_mode(k1)
    rng = np.random.default_rng(7)
    contigs, segs, phase = _random_case(rng, 200)
    tbl = _table(segs, phase, framing=(prep != "defer"))
    want = ref.check(contigs, tbl, 1, ("ATG",), True)
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        if prep == "sync":
            plan.prepare()
        else:
            plan.prepare_async(defer_records=(prep == "defer"))
        for counts in (False, True):
            for junctions in (False, True):
                got = plan.check(None, use_phase=True, codon_usage=counts, junctions=junctions)
                assert (got[1] is None) == (not counts) and (got[2] is None) == (not junctions)
                _assert_same(got, want, contigs, tbl)
        # the device variant into poisoned buffers, every NULL combination
        import torch
        n, e = tbl.n_rec, tbl.n_seg
        for counts in (False, True):
            for junctions in (False, True):
                d_rec = torch.full((n * 56,), 0xA5, dtype=torch.uint8, device="cuda")
                d_cnt = torch.full((n * 256,), 0xA5, dtype=torch.uint8, device="cuda") if counts else None
                d_jn = torch.full((max(e, 1),), 0x7F, dtype=torch.uint8, device="cuda") if junctions else None
                _lib.check(_lib.lib.mg_plan_check_device(plan.handle, _lib.MG_PROT_USE_PHASE, None, ctypes.c_void_p(d_rec.data_ptr()),
                                                         ctypes.c_void_p(d_cnt.data_ptr()) if counts else None,
                                                         ctypes.c_void_p(d_jn.data_ptr()) if junctions else None, None))
                torch.cuda.synchronize()
                recs = d_rec.cpu().numpy().view(engine.CHECK_DTYPE)
                cnt = d_cnt.cpu().numpy().view(np.uint32).reshape(n, 64) if counts else None
                jn = d_jn.cpu().numpy()[:e].view(np.int8) if junctions else None
                _assert_same((recs, cnt, jn), want, contigs, tbl)
        plan.close()
    finally:
        g.close()


@pytest.mark.parametrize("framing", [False, True])
@pytest.mark.parametrize("size", ["tiny", "short"])
def test_many_records_per_tile(mg, size, framing):
    """More than 64 records in a 32 KB tile, so the codon pass stages, searches and flushes them in several batches: thousands
    of 0-9 base records (the tile overflows the piece staging and takes the generic path) or ~120-250 records of 120-300 bases
    (staged pieces, two to four batches)."""
    from magot_b200 import engine
    rng = np.random.default_rng(23)
    alpha = np.frombuffer(b"ACGTACGTACGTacgtNGTAGTAATGA", dtype=np.uint8)
    contigs = [alpha[rng.integers(0, alpha.size, size=200000)].tobytes()]
    segs = []
    pos = 1
    for r in range(6000 if size == "tiny" else 1200):
        m = int(rng.integers(0, 2))
        if size == "tiny":
            ln = int(rng.integers(0, 10))
            row = [(0, pos, pos + ln - 1, m)]
        else:
            a, b = int(rng.integers(60, 150)), int(rng.integers(60, 150))
            row = [(0, pos, pos + a - 1, m), (0, pos + a + int(rng.integers(0, 8)), pos + a + 10 + b, m)]
            if m:
                row.reverse()
        segs.append(row)
        pos += 1 + int(rng.integers(0, 160 if size == "short" else 20))
        pos %= 190000
    phase = rng.integers(0, 3, size=len(segs))
    tbl = _table(segs, phase, framing=framing)
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        plan.prepare()
        for use_phase in (False, True):
            want = ref.check(contigs, tbl, 1, ("ATG", "GTG"), use_phase)
            from magot_b200 import gencode
            _assert_same(plan.check(gencode.start64(("ATG", "GTG")), use_phase, True, True), want, contigs, tbl)
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
        recs = np.zeros(1, dtype=engine.CHECK_DTYPE)
        P = ctypes.c_void_p(recs.ctypes.data)
        assert _lib.lib.mg_plan_check(plan.handle, 0, None, P, None, None, None) == -4      # not prepared
        plan.prepare()
        assert _lib.lib.mg_plan_check(plan.handle, _lib.MG_PROT_TRIMX, None, P, None, None, None) == -1
        assert _lib.lib.mg_plan_check(plan.handle, 0, bytes(64), P, None, None, None) == -1
        assert "no start codon" in _lib.last_error()
        assert _lib.lib.mg_plan_check(plan.handle, 0, gencode.start64(["TAA"], 6), P, None, None, None) == -1
        assert "stop codon" in _lib.last_error()           # TAA is a stop of table 1, the plan's code
        plan.set_codon_table(gencode.codon64(6))            # ... and not of table 6
        assert _lib.lib.mg_plan_check(plan.handle, 0, gencode.start64(["TAA"], 6), P, None, None, None) == 0
        g.mask([0], [3], [6], hard=True)
        assert _lib.lib.mg_plan_check(plan.handle, 0, None, P, None, None, None) == -4      # genome changed
        assert "prepare it again" in _lib.last_error()
        plan.close()
    finally:
        g.close()


def test_agrees_with_protein_text(mg):
    """trimX off: residue i of the protein text is '*' exactly at stop codons and 'X' exactly at ambiguous ones, and the residue
    composition under the code is what the 64 counts give."""
    from magot_b200 import engine, gencode
    rng = np.random.default_rng(3)
    contigs, segs, _ = _random_case(rng, 300)
    tbl = _table(segs, framing=False)
    g = _genome(contigs)
    try:
        for code in (1, 2):
            plan = engine.Plan(g, tbl)
            t64 = gencode.codon64(code)
            if code != 1:
                plan.set_codon_table(t64)
            plan.prepare(trimx=False)
            recs, counts, _ = plan.check(None, codon_usage=True)
            prot = plan.emit_bytes(protein=True)
            _, aa = plan.lengths()
            off = np.concatenate(([0], np.cumsum(np.maximum(aa, 0))))
            for r in range(tbl.n_rec):
                n = int(recs["n_codons"][r])
                p = np.frombuffer(prot[off[r]:off[r + 1]], dtype=np.uint8)[:n]
                assert p.size == n
                assert int((p == ord("X")).sum()) == int(recs["n_ambig"][r])
                assert int((p == ord("*")).sum()) == int(recs["n_stop"][r])
                stops = np.flatnonzero(p == ord("*"))
                assert int(recs["first_stop"][r]) == (int(stops[0]) if stops.size else -1)
                comp = np.bincount(p[(p != ord("X"))], minlength=256)
                want = np.zeros(256, dtype=np.int64)
                np.add.at(want, np.frombuffer(t64, dtype=np.uint8), counts[r].astype(np.int64))
                assert np.array_equal(comp, want)
            plan.close()
    finally:
        g.close()


def test_masks(mg):
    """A soft mask changes nothing; a hard mask makes the codons it touches ambiguous; a check after a mask needs a prepare."""
    from magot_b200 import engine
    rng = np.random.default_rng(11)
    contigs, segs, _ = _random_case(rng, 200)
    contigs = [c.upper() for c in contigs]
    tbl = _table(segs)
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        plan.prepare()
        before = plan.check(None, codon_usage=True, junctions=True)
        lo = np.array([100, 20000, 60000], dtype=np.int64)
        hi = lo + 2500
        cid = np.array([3, 4, 5], dtype=np.int32)
        g.mask(cid, lo, hi, hard=False)
        with pytest.raises(Exception, match="prepare it again"):
            plan.check(None)
        plan.prepare()
        after = plan.check(None, codon_usage=True, junctions=True)
        assert ref.compare(after[0], [dict(zip(engine.CHECK_DTYPE.names, x)) for x in before[0].tolist()]) is None
        assert np.array_equal(before[1], after[1]) and np.array_equal(before[2], after[2])
        g.mask(cid, lo, hi, hard=True)
        plan.prepare()
        hard = [bytearray(c) for c in contigs]
        for c, a, b in zip(cid.tolist(), lo.tolist(), hi.tolist()):
            hard[c][a:b] = b"N" * (b - a)
        hard = [bytes(c) for c in hard]
        _assert_same(plan.check(None, codon_usage=True, junctions=True), ref.check(hard, tbl), hard, tbl)
        plan.close()
    finally:
        g.close()


def test_graph_capture_and_replay(mg):
    import torch
    from magot_b200 import engine, _lib
    L = _lib.lib
    rng = np.random.default_rng(5)
    contigs, segs, phase = _random_case(rng, 300)
    tbl = _table(segs, phase)
    want = ref.check(contigs, tbl, 1, ("ATG",), True)
    g = _genome(contigs)
    s = torch.cuda.Stream()
    sp = ctypes.c_void_p(s.cuda_stream)
    try:
        plan = engine.Plan(g, tbl, stream=sp)
        plan.prepare_async()
        n, e = tbl.n_rec, tbl.n_seg
        d_rec = torch.empty(n * 56, dtype=torch.uint8, device="cuda")
        d_cnt = torch.empty(n * 256, dtype=torch.uint8, device="cuda")
        d_jn = torch.empty(e, dtype=torch.uint8, device="cuda")
        cap_n, cap_p = plan.capacities()
        torch.cuda.synchronize()
        _lib.check(L.mg_graph_begin(0, sp))
        try:
            _lib.check(L.mg_plan_prepare_async(plan.handle, _lib.MG_PROT_DEFER, cap_n, cap_p, sp))
            _lib.check(L.mg_plan_check_device(plan.handle, _lib.MG_PROT_USE_PHASE, None, ctypes.c_void_p(d_rec.data_ptr()),
                                              ctypes.c_void_p(d_cnt.data_ptr()), ctypes.c_void_p(d_jn.data_ptr()), sp))
        finally:
            gx = ctypes.c_void_p()
            _lib.check(L.mg_graph_end(0, sp, ctypes.byref(gx)))
        for _ in range(3):
            d_rec.fill_(0xA5)
            d_cnt.fill_(0x5A)
            d_jn.fill_(0x7F)
            torch.cuda.synchronize()
            _lib.check(L.mg_graph_launch(0, gx, sp))
            s.synchronize()
            got = (d_rec.cpu().numpy().view(engine.CHECK_DTYPE), d_cnt.cpu().numpy().view(np.uint32).reshape(n, 64),
                   d_jn.cpu().numpy().view(np.int8))
            _assert_same(got, want, contigs, tbl)
        _lib.check(L.mg_graph_destroy(gx))
        # the host variant allocates its device outputs on first use: inside a capture that is refused, outside it works
        plan2 = engine.Plan(g, tbl, stream=sp)
        plan2.prepare()
        recs = np.zeros(n, dtype=engine.CHECK_DTYPE)
        torch.cuda.synchronize()
        _lib.check(L.mg_graph_begin(0, sp))
        _lib.check(L.mg_plan_check_device(plan.handle, 0, None, ctypes.c_void_p(d_rec.data_ptr()), None, None, sp))
        rc = L.mg_plan_check(plan2.handle, 0, None, ctypes.c_void_p(recs.ctypes.data), None, None, sp)
        err = _lib.last_error()
        gx = ctypes.c_void_p()
        _lib.check(L.mg_graph_end(0, sp, ctypes.byref(gx)))
        _lib.check(L.mg_graph_destroy(gx))
        assert rc == -4 and "capture" in err
        _assert_same(plan2.check(None, junctions=True), ref.check(contigs, tbl), contigs, tbl)
        plan.close()
        plan2.close()
    finally:
        g.close()


def _stdout_of(fn, *a, **k):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        fn(*a, **k)
    return buf.getvalue()


def test_obiroi_check_cds_tool(mg, tmp_path):
    """The whole tool on the reference's O. biroi RefSeq fixture against the model, and the per-flag record counts pinned."""
    from magot_b200 import genome, genome_tools
    d = os.path.join(HERE, "golden", "ref_test_data")
    fa, gff = tmp_path / "g.fa", tmp_path / "a.gff"
    fa.write_bytes(gzip.open(os.path.join(d, "O.biroi_refseqGenomeSubset.fasta.gz")).read())
    gff.write_bytes(gzip.open(os.path.join(d, "O.biroi_NCBIrefseq_gff3Subset.gff.gz")).read())
    got = _stdout_of(genome_tools.main, ["genome_tools", "check_cds", str(fa), str(gff)])
    g = genome.Genome(str(fa))
    g.read_gff(str(gff))
    res = g.annotations.check_cds("gene")
    # the model from the FASTA bytes and the same record table
    from magot_b200.genome import _native_table, _PENDING
    g2 = genome.Genome(str(fa))
    g2.read_gff(str(gff))
    gs, tbl, _ = _native_table(g2.annotations, _PENDING.get(g2.annotations), "gene")
    names = list(gs)
    contigs = [None] * len(names)
    for n in names:
        contigs[gs.contig_index(n)] = str(gs[n]).encode("latin-1")
    recs, counts, _ = ref.check(contigs, tbl)
    keep = np.flatnonzero(tbl.rec_pre_len > 0)
    want = [dict(r) for r in np.array(recs, dtype=object)[keep]]
    assert ref.compare(res.records, want) is None
    assert got == "\n".join(genome_tools._check_tsv_lines(res.names, res.records)) + "\n"
    # exactly the records of get_fasta(feature, seq_type="protein"), same order, same names
    g3 = genome.Genome(str(fa))
    g3.read_gff(str(gff))
    text = g3.annotations.get_fasta("gene", seq_type="protein")
    assert res.names == [line[1:] for line in text.split("\n") if line.startswith(">")]
    # the object model (the set materialised): the Flattener path gives the same result
    assert len(g3.annotations.gene) > 0
    obj = g3.annotations.check_cds("gene")
    assert obj.names == res.names
    assert ref.compare(obj.records, want) is None
    usage = _stdout_of(genome_tools.main, ["genome_tools", "check_cds", str(fa), str(gff), "out_format=codon_usage"])
    assert usage == "\n".join(genome_tools._codon_usage_lines(counts[keep].sum(axis=0), 1)) + "\n"
    flags = res.records["flags"]
    tally = {name: int(((flags >> k) & 1).sum()) for k, name in enumerate(("NO_START", "NO_STOP", "INTERNAL_STOP", "PARTIAL_CODON",
                                                                            "NONCANONICAL_SPLICE", "AMBIGUOUS", "EMPTY"))}
    tally["ok"] = int((flags == 0).sum())
    tally["records"] = len(res.names)
    print("O. biroi check_cds tally:", tally)
    assert tally == OBIROI_TALLY, tally


#: per-flag record counts of `check_cds` on the O. biroi RefSeq subset (genes, table 1, ATG, no phase)
OBIROI_TALLY = {"NO_START": 0, "NO_STOP": 0, "INTERNAL_STOP": 0, "PARTIAL_CODON": 0, "NONCANONICAL_SPLICE": 3, "AMBIGUOUS": 0,
                "EMPTY": 0, "ok": 82, "records": 85}


def test_large_genome_past_2e31(mg):
    """Records on a contig that starts past forward index 2^31, and '-' records on the first contig, whose reverse-plane
    indices lie past 2^32 (the reverse plane starts at T > 2^31 and holds the first contig at its end)."""
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
        got = plan.check(None, codon_usage=True, junctions=True)
        plan.close()
        contigs = [small[0], filler.tobytes(), small[1]]
        _assert_same(got, ref.check(contigs, tbl), contigs, tbl)
        # segments of 2^31 bases or more, which the plan splits into chunks: junctions are reported per caller segment and
        # the chunk boundaries are none
        long_segs = [[(1, 1, big - 100, 0), (1, big - 90, big - 10, 0)], [(1, big - 90, big - 10, 1), (1, 1, big - 100, 1)],
                     [(0, 1, 500, 0), (1, 1, big, 0), (1, 20, 80, 0)], [(1, -big, -1, 1), (2, 1, 10, 1)]]
        tbl = _table(long_segs)
        plan = engine.Plan(g, tbl)
        plan.prepare_async(defer_records=True)
        recs, _, junc = plan.check(None, junctions=True)
        plan.close()
        want_j = np.array([ref.junction_class(contigs, tbl, e) for e in range(tbl.n_seg)], dtype=np.int8)
        assert np.array_equal(junc, want_j)
        for r in range(tbl.n_rec):
            j = want_j[tbl.rec_seg_off[r]:tbl.rec_seg_off[r + 1]]
            assert int(recs["n_junction"][r]) == int((j > 0).sum()) and int(recs["n_noncanonical"][r]) == int((j == 4).sum())
            ln = sum(b - a for a, b in (ref.clamp(len(contigs[c]), st, en) for c, st, en, _ in long_segs[r]))
            assert int(recs["nuc_len"][r]) == ln and int(recs["n_codons"][r]) == ln // 3
    finally:
        g.close()
