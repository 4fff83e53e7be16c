"""Variant consequences on the device (mg_plan_variant_count / _emit*, engine.Plan.variant_effects, AnnotationSet.variant_effects,
genome_tools variant_effects), row for row and bit for bit against the model variant_ref: random tables with mixed strands and
phases under codes 1, 2 and 11 and three start sets; every SNV of small multi-exon records on both strands; indels and MNVs at
segment edges, across junctions and on the sites; insertions at the points a site shares with its segment; alternative
transcripts sharing exons; each status; gaps under 4 bases; a genome past forward index 2^31 and reverse-plane index 2^32 with
segments the plan splits into chunks; the argument and state errors; and the O. biroi fixture against K2 + mg_translate_ascii_table."""
import ctypes
import os

import numpy as np
import pytest

import gencode_ref as gref
import variant_ref as ref
from test_gpu_check import START_SETS, _genome, _random_case, _starts, _table

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
MG_ESTATE = -4


@pytest.fixture(scope="module")
def mg():
    import magot_b200
    return magot_b200


def _pack(alleles):
    """(contig, pos, allele_off, bytes) arrays of an allele list [(contig, pos, ref, alt)]."""
    contig = np.array([a[0] for a in alleles], dtype=np.int32)
    pos = np.array([a[1] for a in alleles], dtype=np.int64)
    parts = [x for a in alleles for x in (bytes(a[2]), bytes(a[3]))]
    off = np.concatenate(([0], np.cumsum([len(x) for x in parts]))).astype(np.int64)
    return contig, pos, off, b"".join(parts)


def _run(plan, alleles, code=1, starts=("ATG",), use_phase=False):
    from magot_b200 import gencode
    c, p, off, buf = _pack(alleles)
    return plan.variant_effects(c, p, off, buf, gencode.start64(starts, code) if starts != ("ATG",) else None, use_phase)


def _check(got, contigs, tbl, alleles, code=1, starts=("ATG",), use_phase=False):
    st, rows = ref.effects(contigs, tbl, alleles, code, starts, use_phase)
    msg = ref.compare(got[0], got[1], st, rows)
    assert msg is None, msg
    return rows


def _mutate(rng, seq):
    return bytes(b"ACGTacgtN"[int(x)] for x in rng.integers(0, 9, size=len(seq)))


def _alleles_near(rng, contigs, points, n_per=6):
    """Alleles around each (contig, forward position): SNVs, MNVs, insertions and deletions with an anchor base, complex
    alleles, mixed case, a few REF mismatches."""
    out = []
    for c, x in points:
        L = len(contigs[c])
        for _ in range(n_per):
            p = int(x) + int(rng.integers(-4, 4))
            if p < 0 or p >= L:
                continue
            kind = int(rng.integers(0, 6))
            lr = 1 if kind in (0, 2) else int(rng.integers(1, 8))
            lr = min(lr, L - p)
            refb = contigs[c][p:p + lr]
            if rng.random() < 0.3:
                refb = refb.lower()
            if kind == 0:                                  # SNV
                alt = bytes([b"ACGTacgtN"[int(rng.integers(0, 9))]])
            elif kind == 1:                                # MNV
                alt = _mutate(rng, refb)
            elif kind == 2:                                # insertion with its anchor base
                alt = refb + _mutate(rng, b"x" * int(rng.integers(1, 8)))
            elif kind == 3:                                # deletion with its anchor base
                alt = refb[:1]
            elif kind == 4:                                # complex
                alt = _mutate(rng, b"x" * int(rng.integers(1, 9)))
            else:                                          # REF and ALT with a common suffix and prefix around a change
                alt = refb[:1] + _mutate(rng, b"x" * int(rng.integers(0, 4))) + refb[1:]
            if rng.random() < 0.03:
                refb = _mutate(rng, refb)                  # mostly a REF mismatch (status 2)
            out.append((c, p, refb, alt))
    return out


def _edges(contigs, tbl):
    pts = []
    for r in range(tbl.n_rec):
        for _, c, cl, ch, _ in ref.segments(contigs, tbl, r):
            if 0 <= c < len(contigs) and ch > cl:
                pts += [(c, cl), (c, ch), (c, (cl + ch) // 2)]
    return pts


def _sort(alleles):
    return sorted(alleles, key=lambda a: (a[0], a[1]))


@pytest.mark.parametrize("code", (1, 2, 11))
def test_random_tables(mg, code):
    from magot_b200 import engine, gencode
    rng = np.random.default_rng(code)
    contigs, segs, _ = _random_case(rng, 200)
    phase = rng.integers(-1, 4, size=len(segs))
    tbl = _table(segs, phase)
    edges = _edges(contigs, tbl)
    pick = rng.choice(len(edges), size=min(len(edges), 800), replace=False)
    alleles = _alleles_near(rng, contigs, [edges[k] for k in pick], 4)
    for _ in range(1000):                                  # and anywhere
        c = int(rng.integers(0, len(contigs)))
        if len(contigs[c]):
            alleles += _alleles_near(rng, contigs, [(c, int(rng.integers(0, len(contigs[c]))))], 1)
    alleles = _sort(alleles)
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        if code != 1:
            plan.set_codon_table(gencode.codon64(code))
        plan.prepare(trimx=False)
        n_rows = 0
        for k, which in enumerate(START_SETS):
            starts = _starts(code, which)
            use_phase = k % 2 == 1
            n_rows = len(_check(_run(plan, alleles, code, starts, use_phase), contigs, tbl, alleles, code, starts, use_phase))
        assert n_rows > 1000
        plan.close()
    finally:
        g.close()


def _small_records():
    """Two contigs with multi-exon records on both strands, alternative transcripts sharing exons, a gap under 4 bases, a
    junction across a contig change and an exon of 1 base."""
    rng = np.random.default_rng(5)
    c0 = bytearray(b"ACGT"[int(x)] for x in rng.integers(0, 4, size=900))
    c0[10:13], c0[167:170] = b"ATG", b"TAG"                 # record 0 starts with ATG and ends with a stop
    contigs = [bytes(c0), bytes(b"ACGTacgt"[int(x)] for x in rng.integers(0, 8, size=700))]
    segs = [
        [(0, 11, 40, 0), (0, 61, 100, 0), (0, 141, 170, 0)],        # '+', three exons
        [(0, 141, 170, 1), (0, 61, 100, 1), (0, 11, 40, 1)],        # the same exons on '-'
        [(0, 11, 40, 0), (0, 141, 170, 0)],                         # an alternative transcript skipping exon 2
        [(0, 201, 230, 0), (0, 233, 260, 0)],                       # a gap of 2 bases: no sites
        [(0, 320, 350, 1), (0, 301, 316, 1)],                       # '-' with a gap of 3 bases: no sites
        [(0, 401, 430, 0), (0, 435, 435, 0), (0, 441, 470, 0)],     # a 1-base exon with 4-base introns around it
        [(0, 501, 540, 0), (1, 11, 50, 0)],                         # a contig change: no sites
        [(1, 101, 150, 1), (1, 61, 80, 1)],                         # '-' on mixed case
    ]
    return contigs, segs


@pytest.mark.parametrize("use_phase", [False, True])
def test_every_snv_of_small_records(mg, use_phase):
    from magot_b200 import engine
    contigs, segs = _small_records()
    tbl = _table(segs, [0, 1, 2, 0, 1, 2, 0, 1])
    alleles = []
    for r in range(tbl.n_rec):
        for _, c, cl, ch, _ in ref.segments(contigs, tbl, r):
            for x in range(max(0, cl - 3), min(len(contigs[c]), ch + 3)):
                for b in b"ACGT":
                    if b != contigs[c][x] & 0xDF:
                        alleles.append((c, x, contigs[c][x:x + 1], bytes([b])))
    alleles = _sort(set(alleles))
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        plan.prepare()
        rows = _check(_run(plan, alleles, use_phase=use_phase), contigs, tbl, alleles, use_phase=use_phase)
        assert {r["cls"] for r in rows} >= ({1, 2, 7, 8, 9, 11, 12} if not use_phase else {1, 2, 7, 8, 11, 12})
        plan.close()
    finally:
        g.close()


def test_indels_mnvs_and_insertions_at_sites(mg):
    from magot_b200 import engine
    contigs, segs = _small_records()
    tbl = _table(segs)
    rng = np.random.default_rng(11)
    alleles = _alleles_near(rng, contigs, _edges(contigs, tbl), 30)
    for r in range(tbl.n_rec):                             # an insertion at every point from cl - 3 to ch + 3
        for _, c, cl, ch, _ in ref.segments(contigs, tbl, r):
            for s in list(range(cl - 3, cl + 4)) + list(range(ch - 3, ch + 4)):
                if 1 <= s <= len(contigs[c]):
                    anchor = contigs[c][s - 1:s]
                    for ins in (b"A", b"GC", b"TTA", b"acgt"):
                        alleles.append((c, s - 1, anchor, anchor + ins))
    alleles = _sort(set(alleles))
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        plan.prepare()
        rows = _check(_run(plan, alleles), contigs, tbl, alleles)
        assert {r["cls"] for r in rows} >= set(range(1, 13))
        per = {}
        for r in rows:
            per.setdefault(r["var"], set()).add(r["rec"])
        assert max(len(v) for v in per.values()) >= 3      # shared exons: one allele, several records
        plan.close()
    finally:
        g.close()


def test_status_cases_and_empty_inputs(mg):
    from magot_b200 import engine, _lib
    contigs = [b"ACGTACGTNNacgtRYKM" * 20, b"GATTACA" * 30 + b"SSWW" + b"GATTACA" * 10]
    tbl = _table([[(0, 3, 60, 0), (0, 70, 120, 0)], [(1, 2, 200, 1)]])
    alleles = _sort([
        (-1, 5, b"A", b"C"), (2, 5, b"A", b"C"), (0, -1, b"A", b"C"), (0, 358, b"KMA", b"A"),   # status 1
        (0, 4, b"T", b"C"), (0, 8, b"n", b"A"), (0, 14, b"r", b"A"), (1, 210, b"S", b"A"),      # 2, 0, 0 (R), 2 (exception)
        (0, 20, b"", b"A"), (0, 21, b"C", b""), (0, 22, b"GT", b"gt"),                          # status 3
        (0, 10, b"acgt", b"aggt"), (1, 3, b"TTACA", b"TT"),
    ])
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        plan.prepare()
        got = _run(plan, alleles)
        _check(got, contigs, tbl, alleles)
        assert sorted(set(got[0].tolist())) == [0, 1, 2, 3]
        st, rows = plan.variant_effects(np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(1, np.int64), b"")
        assert st.size == 0 and rows.size == 0
        plan.close()
        empty = engine.Plan(g, _table([]))
        empty.prepare()
        st, rows = _run(empty, alleles)
        assert rows.size == 0 and st.tolist() == ref.effects(contigs, _table([]), alleles)[0]
        empty.close()
    finally:
        g.close()


def test_argument_and_state_errors(mg):
    from magot_b200 import engine, _lib
    contigs, segs = _small_records()
    tbl = _table(segs)
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        rows = np.zeros(64, dtype=engine.VEF_DTYPE)
        emit = lambda: _lib.lib.mg_plan_variant_emit(plan.handle, ctypes.c_void_p(rows.ctypes.data), None)
        alleles = [(0, 15, contigs[0][15:16], b"N"), (0, 70, contigs[0][70:71], b"T" if contigs[0][70] != ord("T") else b"A")]
        with pytest.raises(_lib.MagotError, match="error -4"):
            _run(plan, alleles)                            # not prepared
        plan.prepare()
        assert emit() == MG_ESTATE                    # no count yet
        with pytest.raises(_lib.MagotError, match="error -1"):
            _run(plan, alleles[::-1])                      # unsorted
        _run(plan, alleles)
        c, p, off, buf = _pack(alleles)
        n = ctypes.c_int64(0)
        st = np.zeros(2, np.int8)
        _lib.check(_lib.lib.mg_plan_variant_count(plan.handle, 2, ctypes.c_void_p(c.ctypes.data), ctypes.c_void_p(p.ctypes.data),
                                                  ctypes.c_void_p(off.ctypes.data), buf, len(buf), 0, None,
                                                  ctypes.c_void_p(st.ctypes.data), ctypes.byref(n), None))
        assert 0 < n.value <= rows.size
        assert emit() == 0
        plan.prepare()
        assert emit() == MG_ESTATE                    # re-prepared since the count
        _run(plan, alleles)
        g.mask(np.array([1], np.int32), np.array([0]), np.array([5]))
        assert emit() == MG_ESTATE                    # genome masked since the count
        with pytest.raises(_lib.MagotError):
            plan.variant_effects(c, p, off, buf, b"\x00" * 64)   # no start codon
        plan.close()
    finally:
        g.close()


def test_device_emit_matches_host_emit(mg):
    import torch
    from magot_b200 import engine, _lib
    contigs, segs = _small_records()
    tbl = _table(segs)
    rng = np.random.default_rng(2)
    alleles = _sort(set(_alleles_near(rng, contigs, _edges(contigs, tbl), 5)))
    g = _genome(contigs)
    try:
        plan = engine.Plan(g, tbl)
        plan.prepare()
        st, rows = _run(plan, alleles)
        d = torch.full((rows.size * 64,), 0xA5, dtype=torch.uint8, device="cuda")
        _lib.check(_lib.lib.mg_plan_variant_emit_device(plan.handle, ctypes.c_void_p(d.data_ptr()), None))
        torch.cuda.synchronize()
        assert d.cpu().numpy().tobytes() == rows.tobytes()
        plan.close()
    finally:
        g.close()


def test_large_genome_past_2e31(mg):
    """Records on a contig that starts past forward index 2^31, '-' records whose reverse-plane indices lie past 2^32, and
    segments of 2^31 bases or more, which the plan splits into chunks: rows stay per caller segment."""
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
    small = [bytes(b"ACGTacgt"[int(x)] for x in rng.integers(0, 8, size=300000)) for _ in range(2)]
    g = engine.DeviceGenome([len(small[0]), big, len(small[1])], device=0)
    try:
        g.pack(0, np.frombuffer(small[0], dtype=np.uint8))
        g.pack(1, filler)
        g.pack(2, np.frombuffer(small[1], dtype=np.uint8))
        g.finalize()
        contigs = [small[0], filler.tobytes(), small[1]]
        segs = []
        for r in range(200):
            c = 2 if r % 2 else 0
            m = (r // 2) % 2
            pos = int(rng.integers(1, 290000))
            row = []
            for _ in range(int(rng.integers(1, 6))):
                ln = int(rng.integers(1, 300))
                row.append((c, pos, min(pos + ln - 1, 299999), m))
                pos += ln + int(rng.integers(0, 40))
            segs.append(row[::-1] if m else row)
        segs += [[(1, 1, big - 100, 0), (1, big - 90, big - 10, 0)], [(1, big - 90, big - 10, 1), (1, 1, big - 100, 1)],
                 [(0, 1, 500, 0), (1, 1, big, 0), (1, 20, 80, 0)], [(1, -big, -1, 1), (2, 1, 10, 1)],
                 [(1, big - 5000, big, 1), (2, 1, 3000, 1)]]
        tbl = _table(segs)
        pts = _edges(contigs, tbl) + [(1, x) for x in (5, 1 << 31, (1 << 31) + 7, big - 95, big - 12, big - 2)]
        alleles = _sort(set(_alleles_near(rng, contigs, pts, 6)))
        plan = engine.Plan(g, tbl)
        plan.prepare()
        rows = _check(_run(plan, alleles), contigs, tbl, alleles)
        assert any(r["rec"] >= 200 for r in rows)
        plan.close()
    finally:
        g.close()


def _translate(texts):
    """mg_translate_ascii_table of each text under code 1, frame 0, no trimX."""
    from magot_b200 import _lib, gencode
    buf = b"".join(texts)
    off = np.concatenate(([0], np.cumsum([len(t) for t in texts]))).astype(np.int64)
    cap = len(buf) // 3 + len(texts) + 16
    out = np.zeros(cap, np.uint8)
    out_off = np.zeros(len(texts) + 1, np.int64)
    out_len = np.zeros(len(texts), np.int64)
    _lib.check(_lib.lib.mg_translate_ascii_table(0, gencode.codon64(1), buf, ctypes.c_void_p(off.ctypes.data), len(texts), 0, 0, 0,
                                                 ctypes.c_void_p(out.ctypes.data), cap, ctypes.c_void_p(out_off.ctypes.data),
                                                 ctypes.c_void_p(out_len.ctypes.data), None))
    return [out[out_off[k]:out_off[k] + max(0, out_len[k])].tobytes() for k in range(len(texts))]


def test_obiroi_snvs_and_tool(mg, tmp_path):
    """SNVs planted in the CDS records of the O. biroi RefSeq fixture: each row's residues and class agree with the record's K2
    text, edited and translated by mg_translate_ascii_table; then genome_tools variant_effects in both formats."""
    import contextlib
    import gzip
    import io
    from magot_b200 import engine, genome, genome_tools
    d = os.path.join(HERE, "golden", "ref_test_data")
    fa, gff = tmp_path / "g.fa", tmp_path / "a.gff"
    fa.write_bytes(gzip.open(os.path.join(d, "O.biroi_refseqGenomeSubset.fasta.gz")).read())
    gff.write_bytes(gzip.open(os.path.join(d, "O.biroi_NCBIrefseq_gff3Subset.gff.gz")).read())
    g = genome.Genome(str(fa))
    g.read_gff(str(gff))
    gs, tbl = genome._feature_table(g.annotations, "gene", "protein")
    names = list(gs)
    contigs = [None] * len(names)
    for n in names:
        contigs[gs.contig_index(n)] = str(gs[n]).encode("latin-1")
    plan = engine.Plan(gs._engine().primary, tbl)
    plan.prepare(trimx=False)
    text = plan.emit_bytes()
    nuc, _ = plan.lengths()
    plan.close()
    frame = tbl.rec_pre_len.astype(np.int64) + tbl.rec_suf_len + nuc
    start = np.concatenate(([0], np.cumsum(frame)))[:-1] + tbl.rec_pre_len
    keep = np.flatnonzero(tbl.rec_pre_len > 0)
    rng = np.random.default_rng(29)
    planted = {}
    for r in keep.tolist():
        segs = ref.segments(contigs, tbl, r)
        L = int(nuc[r])
        for q in rng.integers(0, max(1, L - L % 3), size=3).tolist():
            o = 0
            for _, c, cl, ch, minus in segs:
                if o <= q < o + ch - cl:
                    x = ch - 1 - (q - o) if minus else cl + q - o
                    b = contigs[c][x:x + 1].upper()
                    if b in (b"A", b"C", b"G", b"T"):
                        planted[(names[c], x + 1)] = (b, bytes([b"ACGT".replace(b, b"")[int(rng.integers(0, 3))]]))
                    break
                o += ch - cl
    order = sorted(planted, key=lambda k: (gs.contig_index(k[0]), k[1]))
    vcf = ["##fileformat=VCFv4.2", "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO"]
    vcf += ["%s\t%d\tv%d\t%s\t%s\t.\tPASS\t." % (k[0], k[1], i, planted[k][0].decode(), planted[k][1].decode()) for i, k in enumerate(order)]
    vcf_path = tmp_path / "calls.vcf"
    vcf_path.write_text("\n".join(vcf) + "\n")
    res = g.annotations.variant_effects("gene", str(vcf_path))
    assert res.status.tolist() == [0] * len(order)
    rec_names = genome._record_names(tbl, keep)
    assert res.names == rec_names
    checked = 0
    for k in range(res.rows.size):
        row = res.rows[k]
        cls = int(row["cls"])
        if not 7 <= cls <= 12:
            continue
        r = int(keep[int(row["rec"])])
        S = text[start[r]:start[r] + nuc[r]]
        a = res.variants.alt[int(row["var"])]
        if res.strand[k]:
            a = gref.revcomp(a)
        lo = int(row["nuc_lo"])
        S2 = S[:lo] + a + S[lo + 1:]
        p1, p2 = _translate([S, S2])
        i = int(row["codon"])
        assert bytes(row["ref_aa"]) == p1[i:i + 1] and bytes(row["alt_aa"]) == p2[i:i + 1]
        if cls == 12:
            assert p1[i] == p2[i]
        elif cls == 11:
            assert p1[i] != p2[i] and p2[i:i + 1] != b"*"
        elif cls == 8:
            assert p2[i:i + 1] == b"*" and p1[i:i + 1] != b"*"
        elif cls == 9:
            assert p1[i:i + 1] == b"*" and i == len(p1) - 1
        elif cls == 7:
            assert i == 0 and S[:3].upper() == b"ATG" and S2[:3].upper() != b"ATG"
        checked += 1
    assert checked >= len(keep)

    def run(fmt):
        buf, err = io.StringIO(), io.StringIO()
        with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(err):
            genome_tools.main(["genome_tools", "variant_effects", str(fa), str(gff), str(vcf_path), "out_format=" + fmt])
        assert "status ok %d" % len(order) in err.getvalue()
        return buf.getvalue().split("\n")

    tsv = run("tsv")
    assert tsv[0] == genome_tools.VARIANT_TSV_HEADER and tsv[-1] == "" and len(tsv) == res.rows.size + 2
    out = run("vcf")[:-1]
    assert out[0] == vcf[0] and out[1] == genome_tools.VARIANT_INFO_HEADER and len(out) == len(vcf) + 1
    with_info = 0
    for a, b in zip(vcf[1:], out[2:]):
        ca, cb = a.split("\t"), b.split("\t")
        assert ca[:7] == cb[:7] and len(ca) == len(cb)
        with_info += ca[7] != cb[7]
        assert ca[7] == cb[7] or cb[7].startswith("MGCSQ=")
    assert with_info == len(set(res.rows["var"].tolist()))
