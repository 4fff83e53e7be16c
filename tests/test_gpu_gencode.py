"""NCBI genetic codes on the device, bit-exact against the oracle (magot_oracle.translate(library=...)) and its numpy
restatement for long contigs (gencode_ref): Sequence.translate / get_orfs, the plan path (K3, K23, the one-launch emit),
gff2fasta / cds2pep / dna2orfs and the K4 six-frame scan with every distinct stop set."""
import contextlib
import gzip
import io
import os

import numpy as np
import pytest

import coracle
import gencode_ref as ref
import magot_oracle as mo
from cksum import cksum

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PLAN_CODES = (1, 2, 5, 6, 22, 23)


@pytest.fixture(scope="module")
def mg():
    import magot_b200
    return magot_b200


def _stdout_of(fn, *a, **k):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        fn(*a, **k)
    return buf.getvalue()


def _t64(code):
    from magot_b200 import gencode
    return gencode.codon64(code).decode()


# ---- Sequence.translate / get_orfs ------------------------------------------------------------------------------------

def test_translate_every_code(mg):
    from magot_b200 import gencode
    rng = np.random.default_rng(1)
    alpha = np.frombuffer(b"ACGTACGTACGTacgtNnRYKM-", dtype=np.uint8)
    seqs = [alpha[rng.integers(0, alpha.size, size=int(n))].tobytes().decode() for n in rng.integers(0, 300, size=40)]
    for code in gencode.SUPPORTED:
        lib = gencode.library(code)
        for s in seqs:
            for frame in (0, 1, 2):
                for strand in "+-":
                    for trim in (True, False):
                        got = mg.Sequence(s).translate(frame=frame, strand=strand, trimX=trim, genetic_code=code)
                        assert got == mg.Sequence(s).translate(library=lib, frame=frame, strand=strand, trimX=trim)
                        assert got == mo.translate(s, frame=frame, strand=strand, trimX=trim, library=lib), (code, s, frame, strand)


def test_kats_through_table_one(mg, kat):
    from magot_b200 import gencode
    for s, frame, strand, trimx, r in kat["translate"]:
        if r == "!IndexError":
            continue
        assert mg.Sequence(s).translate(frame=frame, strand=strand, trimX=trimx, genetic_code=1) == r
        assert mg.Sequence(s).translate(frame=frame, strand=strand, trimX=trimx, library=gencode.library(1)) == r
    for s, mode, r in kat["get_orfs"][:90]:
        if mode == "longest":
            if r != "!IndexError":
                assert mg.Sequence(s).get_orfs(longest=True, genetic_code=1) == r
        else:
            assert mg.Sequence(s).get_orfs(from_atg=mode, genetic_code="1") == r


def test_get_orfs_other_codes(mg):
    from magot_b200 import gencode
    rng = np.random.default_rng(2)
    for code in (2, 5, 6, 23):
        for n in (0, 3, 10, 200, 901):
            s = "".join(rng.choice(list("ACGTacgtN"), size=n))
            for atg in (False, True):
                assert mg.Sequence(s).get_orfs(from_atg=atg, genetic_code=code) == ref.get_orfs(s, gencode.library(code), from_atg=atg)


# ---- plan path --------------------------------------------------------------------------------------------------------

def _random_plan_case(rng):
    alpha = np.frombuffer(b"ACGTACGTACGTacgtacgtNnRYKM-*xS", dtype=np.uint8)
    contigs = [alpha[rng.integers(0, alpha.size, size=int(n))].copy() for n in (0, 3, 1000, 40000, 70000)]
    n_rec = 300
    n_seg = rng.integers(0, 13, size=n_rec)
    rec_off = np.concatenate(([0], np.cumsum(n_seg)))
    E = int(rec_off[-1])
    cid = rng.integers(0, len(contigs), size=E).astype(np.int32)
    L = np.array([a.size for a in contigs], dtype=np.int64)[cid]
    st = rng.integers(-20, L + 30)
    en = st + rng.integers(-5, 700, size=E)
    st, en = np.minimum(st, en), np.maximum(st, en)
    sd = rng.integers(0, 2, size=E).astype(np.int8)
    segs = [[(int(cid[e]), int(st[e]), int(en[e]), int(sd[e])) for e in range(rec_off[r], rec_off[r + 1])] for r in range(n_rec)]
    return contigs, segs


def _edge_case():
    contig = np.frombuffer(b"ACGTNNacgtTTGACCATGGGTAAACTGATCGATCGTAGCTAGCTAGCTAGCATCGATCGATAGAAGGTCATTAtga" * 3, dtype=np.uint8)
    L = contig.size
    recs = [[], [(5, 4, 0)], [(1, 1, 0)], [(1, 2, 1)], [(1, 3, 1)], [(L, L, 1), (1, 1, 0)], [(L - 1, L + 50, 0)], [(L + 5, L + 9, 0)],
            [(1, L, 1)], [(2, 1, 0), (3, 2, 0), (10, 30, 0)], [(1, 3, 0)] * 40, [(7, 7, 1)] * 33, [(1, L, 0)]]
    return [contig.copy()], [[(0, a, b, m) for (a, b, m) in r] for r in recs]


def _tiny_case(rng):
    alpha = np.frombuffer(b"ACGTacgtNnRY*", dtype=np.uint8)
    contigs = [alpha[rng.integers(0, alpha.size, size=n)].copy() for n in (50_000, 777, 120_000)]
    segs = []
    for r in range(1500):
        k = 400 if r % 50 == 0 else int(rng.integers(0, 40))
        row = []
        for _ in range(k):
            c = int(rng.integers(0, 3))
            a = int(rng.integers(1, contigs[c].size - 10))
            row.append((c, a, a + int(rng.integers(0, 8)), int(rng.integers(0, 2))))
        segs.append(row)
    return contigs, segs


def _table(segs, framing):
    from magot_b200 import engine
    rec_off = np.concatenate(([0], np.cumsum([len(r) for r in segs]))).astype(np.int64)
    flat = [x for r in segs for x in r]
    cid = np.array([x[0] for x in flat], dtype=np.int32)
    st = np.array([x[1] for x in flat], dtype=np.int64)
    en = np.array([x[2] for x in flat], dtype=np.int64)
    sd = np.array([x[3] for x in flat], dtype=np.int8)
    n = len(segs)
    names = [b">r%d\n" % i for i in range(n)]
    if framing:
        pre = np.array([len(x) for x in names], dtype=np.int32)
        suf = np.ones(n, dtype=np.int32)
        lit = np.frombuffer(b"".join(x + b"\n" for x in names), dtype=np.uint8)
    else:
        pre = suf = np.zeros(n, dtype=np.int32)
        lit = np.zeros(0, dtype=np.uint8)
    lit_off = np.concatenate(([0], np.cumsum(pre.astype(np.int64) + suf)[:-1])) if n else np.zeros(0, np.int64)
    return engine.RecordTable(rec_off, cid, st, en, sd, lit_off, pre, suf, lit), names


def _expected(contigs, segs, names, framing, code):
    """Oracle texts: the spliced nucleotides of every record (Python slice rules) and their translation under `code`."""
    texts = [c.tobytes() for c in contigs]
    nuc, prot = [], []
    for r, row in enumerate(segs):
        s = b""
        for (c, a, b, m) in row:
            piece = texts[c][slice(a - 1, b)]
            s += ref.revcomp(piece) if m else piece
        t = ref.translate(s, _t64(code)) or b""
        head, tail = (names[r], b"\n") if framing else (b"", b"")
        nuc.append(head + s + tail)
        prot.append(head + t + tail)
    return b"".join(nuc), b"".join(prot)


def _genome(contigs):
    from magot_b200 import engine
    g = engine.DeviceGenome([a.size for a in contigs], device=0)
    for i, a in enumerate(contigs):
        g.pack(i, a)
    g.finalize()
    return g


def _plan_variants(g, tbl, code, want_n, want_p):
    """K3 (host + device), K23 (after prepare and prepare_async), the one-launch emit, MG_PROT_DEFER."""
    import torch
    from magot_b200 import engine, gencode
    t = None if code is None else gencode.codon64(code)
    text, _ = engine.run_table(g, tbl, protein=True, codon64=t)
    assert text == want_p, "K3 host"
    for async_prepare in (False, True):
        n, p = engine.run_table_both(g, tbl, async_prepare=async_prepare, codon64=t)
        assert n == want_n and p == want_p, ("K23", async_prepare)
    a, bn, bp = engine.run_products(g, tbl, tbl, codon64=t)
    assert a == want_n and bn == want_n and bp == want_p, "one-launch emit"
    for defer in (False, True):
        plan = engine.Plan(g, tbl)
        if t is not None:
            plan.set_codon_table(t)
        cap_n, cap_p = plan.capacities()
        plan.prepare_async(cap_n, cap_p, defer_records=defer)
        if defer:
            plan.prepare_prot()
        out_n = torch.zeros((cap_n + 31) // 32 * 32 + 32, dtype=torch.uint8, device="cuda")
        out_p = torch.zeros((cap_p + 31) // 32 * 32 + 32, dtype=torch.uint8, device="cuda")
        plan.emit_device(out_p.data_ptr(), protein=True)
        plan.emit_device(out_n.data_ptr(), protein=False)
        nt, pt = plan.totals()
        assert out_p[:pt].cpu().numpy().tobytes() == want_p, ("K3 device after prepare_async", defer)
        assert out_n[:nt].cpu().numpy().tobytes() == want_n
        plan.close()


@pytest.mark.parametrize("case", ["random", "edge", "tiny", "twin"])
def test_plan_path_codes(mg, case):
    from magot_b200 import engine, synth
    rng = np.random.default_rng(11)
    framing = case in ("random", "twin")
    if case == "twin":                                     # synthetic twin of config 3
        layout = synth.contig_layout("insect", 2_000_000, 3)
        contigs = synth.synth_genome_host(layout, 3, n_mean=300)
        ann = synth.synth_annotation(layout, 800, 3)
        t = ann.table("cds", framing=False)
        segs = [[(int(t.seg_contig[e]), int(t.seg_start[e]), int(t.seg_end[e]), int(t.seg_strand[e]))
                 for e in range(t.rec_seg_off[r], t.rec_seg_off[r + 1])] for r in range(t.n_rec)]
    else:
        contigs, segs = {"random": lambda: _random_plan_case(rng), "edge": _edge_case, "tiny": lambda: _tiny_case(rng)}[case]()
    g = _genome(contigs)
    tbl, names = _table(segs, framing)
    default_p = engine.run_table(g, tbl, protein=True)[0]
    for code in PLAN_CODES:
        want_n, want_p = _expected(contigs, segs, names, framing, code)
        if code == 1:
            assert want_p == default_p
            _plan_variants(g, tbl, None, want_n, want_p)
        _plan_variants(g, tbl, code, want_n, want_p)
    # one plan: set a code, reset it -- the default bytes come back
    plan = engine.Plan(g, tbl)
    plan.prepare()
    from magot_b200 import gencode
    plan.set_codon_table(gencode.codon64(2))
    assert plan.emit_bytes(protein=True) == _expected(contigs, segs, names, framing, 2)[1]
    plan.set_codon_table(None)
    assert plan.emit_bytes(protein=True) == default_p
    plan.close()
    g.close()


# ---- gff2fasta / cds2pep ----------------------------------------------------------------------------------------------

def _records(text):
    recs = []
    for block in text.split(">")[1:]:
        head, _, body = block.partition("\n")
        recs.append((head, body.rstrip("\n")))
    return recs


@pytest.mark.parametrize("pair", ["obiroi", "c14"])
def test_gff2fasta_genetic_code(mg, ref_data, manifest, pair):
    from magot_b200 import genome_tools as gt, gencode
    if pair == "obiroi":
        fa = os.path.join(ref_data, "O.biroi_refseqGenomeSubset.fasta")
        gff = os.path.join(ref_data, "O.biroi_NCBIrefseq_gff3Subset.gff")
        key = "obiroi:gff2fasta_protein"
    else:
        fa, gff = os.path.join(ref_data, "C14.fasta"), os.path.join(ref_data, "StandardGTF.gtf")
        key = "suite:gff2fasta_C14_StandardGTF_protein"
    p1 = _stdout_of(gt.main, ["genome_tools.py", "gff2fasta", fa, gff, "seq_type=protein", "genetic_code=1"])
    assert cksum(p1) == (manifest[key]["cksum"], manifest[key]["bytes"])
    if pair == "obiroi":
        with gzip.open(os.path.join(GOLDEN, "obiroi_gff2fasta_protein.fa.gz"), "rb") as fh:
            assert p1.encode("latin-1") == fh.read()
    nuc = _records(_stdout_of(gt.gff2fasta, fa, gff))
    for code in (5, 2):
        got = _records(_stdout_of(gt.main, ["genome_tools.py", "gff2fasta", fa, gff, "seq_type=protein", "genetic_code=%d" % code]))
        assert [h for h, _ in got] == [h for h, _ in nuc]
        for (h, p), (_, n) in zip(got, nuc):
            assert p == (mo.translate(n, library=gencode.library(code)) or ""), (code, h)
        assert got != _records(p1)


def test_cds2pep_genetic_code(mg, ref_data):
    from magot_b200 import genome_tools as gt, gencode
    path = os.path.join(ref_data, "CDSannotations.cds")
    got = _stdout_of(gt.main, ["genome_tools.py", "cds2pep", path, "genetic_code=2"])
    lib = gencode.library(2)
    headers, seqs, cur = [], [], None
    with open(path, encoding="latin-1", newline="\n") as fh:
        for line in fh:
            line = line.rstrip("\n").rstrip("\r")
            if line.startswith(">"):
                if cur is not None:
                    seqs.append("".join(cur))
                headers.append(line)
                cur = []
            else:
                cur.append(line)
    seqs.append("".join(cur))
    want = "".join(h + "\n" + str(mo.translate(s, library=lib)) + "\n" for h, s in zip(headers, seqs))
    assert got == want


# ---- K4 ---------------------------------------------------------------------------------------------------------------

def _k4_contigs(rng, code):
    """Contigs of every awkward length, stop-free A/C stretches over several tiles, and N / IUPAC / lower case written over
    stop codons of `code` on both strands."""
    alpha = np.frombuffer(b"ACGTacgtNnR", dtype=np.uint8)
    p = np.array([30, 30, 30, 30, 10, 10, 10, 10, 2, 1, 1], dtype=float)
    out = []
    for n in [0, 1, 2, 3, 4, 5, 6, 7, 8, 24575, 24576, 24577, 73727, 73728, 73729, 147455, 147457, 200001]:
        out.append(alpha[rng.choice(alpha.size, size=n, p=p / p.sum())].tobytes())
    ac = np.frombuffer(b"AC", dtype=np.uint8)
    c = bytearray(alpha[rng.integers(0, 4, size=400000)].tobytes())
    c[60000:300000] = ac[rng.integers(0, 2, size=240000)].tobytes()
    out.append(bytes(c))
    out.append(ac[rng.integers(0, 2, size=73728 * 2 + 5)].tobytes())
    stops = [s.encode() for s, a in ref.library(code).items() if a == "*"]
    c = bytearray(alpha[rng.integers(0, 4, size=30000)].tobytes())
    for k in range(0, 30000 - 3, 7):
        s = stops[k % len(stops)] if stops else b"TAA"
        if (k // 7) % 2:
            s = ref.revcomp(s)
        v = int(rng.integers(0, 4))
        if v == 1:
            s = s.lower()
        elif v == 2:
            s = s[:1] + b"N" + s[2:]
        elif v == 3:
            s = s[:2] + b"Y"
        c[k:k + 3] = s
    out.append(bytes(c))
    return out


def _k4_expected(contigs, min_aa, code):
    per = []
    for c in contigs:
        a, r = ref.sixframe(c, min_aa, _t64(code))
        per.append((a, r))
    return per


def _k4_check(recs, aa, ids, per):
    assert aa == b"".join(per[c][0] for c in ids)
    want = [(c,) + row for c in ids for row in per[c][1]]
    got = [(int(r["contig"]), int(r["frame"]), int(r["minus"]), int(r["start"]), int(r["len"])) for r in recs]
    assert got == want


@pytest.fixture()
def six_mode(mg):
    from magot_b200 import _lib
    yield lambda v: _lib.check(_lib.lib.mg_tune(b"six", v))
    _lib.check(_lib.lib.mg_tune(b"six", 2))


@pytest.mark.parametrize("code", ref.STOP_SET_CODES)
def test_sixframe_stop_sets(mg, six_mode, code, monkeypatch):
    from magot_b200 import orfs
    rng = np.random.default_rng(500 + code)
    contigs = _k4_contigs(rng, code)
    g = _genome([np.frombuffer(c, dtype=np.uint8) for c in contigs])
    n = len(contigs)
    for min_aa in (0, 1, 16, 95, 96, 100, 300):
        per = _k4_expected(contigs, min_aa, code)
        for mode in ((2, 1, 0) if min_aa >= 96 else (2,)):
            six_mode(mode)
            recs, aa = orfs.sixframe(g, 0, n, min_aa, genetic_code=code)
            _k4_check(recs, aa, list(range(n)), per)
        six_mode(2)
        ids = [n - 1, 3, n - 3, 0, 18, 18, 12]
        recs, aa = orfs.sixframe_list(g, ids, min_aa, genetic_code=code)
        _k4_check(recs, aa, ids, per)
    monkeypatch.setenv("MG_SIX_HIT_CAP", "7")            # the dense second pass (k_six_orfs<true>)
    for min_aa in (0, 16):
        per = _k4_expected(contigs[:19], min_aa, code)
        recs, aa = orfs.sixframe(g, 0, 19, min_aa, genetic_code=code)
        _k4_check(recs, aa, list(range(19)), per)
    g.close()


def test_stop_index_cache(mg):
    """Table 1 -> 2 -> 1 -> 6 on one genome, then mask, then table 1: every result equals that of a freshly packed genome, and
    a non-default scan leaves the table-1 result byte-identical.  The second index is counted in device_bytes."""
    from magot_b200 import engine, orfs
    rng = np.random.default_rng(9)
    contigs = [rng.choice(np.frombuffer(b"ACGTacgtN", dtype=np.uint8), size=n) for n in (300000, 73729, 5000)]

    def fresh(code, masked=False):
        cs = [c.copy() for c in contigs]
        if masked:
            cs[0][1000:90000] = ord("N")
        h = _genome(cs)
        r = orfs.sixframe(h, 0, 3, 100, genetic_code=code)
        h.close()
        return r

    def same(a, b):
        return a[1] == b[1] and np.array_equal(a[0], b[0])

    g = _genome(contigs)
    b0 = g.device_bytes()
    r1 = orfs.sixframe(g, 0, 3, 100)
    b1 = g.device_bytes()
    assert same(r1, fresh(1))
    assert same(orfs.sixframe(g, 0, 3, 100, genetic_code=2), fresh(2))
    b2 = g.device_bytes()
    assert b1 > b0 and b2 - b1 == b1 - b0                # one more index of the same size
    assert same(orfs.sixframe(g, 0, 3, 100, genetic_code=1), r1)
    assert same(orfs.sixframe(g, 0, 3, 100, genetic_code=6), fresh(6))
    assert g.device_bytes() == b2                        # at most one non-default index
    g.mask([0], [1000], [90000], hard=True)
    assert same(orfs.sixframe(g, 0, 3, 100, genetic_code=1), fresh(1, masked=True))
    assert same(orfs.sixframe(g, 0, 3, 100, genetic_code=6), fresh(6, masked=True))
    g.close()


@pytest.mark.parametrize("from_atg,longest", [(False, False), (True, False), (False, True)])
def test_dna2orfs_genetic_code(mg, tmp_path, from_atg, longest):
    from magot_b200 import genome_tools as gt, gencode
    rng = np.random.default_rng(7)
    seqs = {"s1": "".join(rng.choice(list("ACGT"), size=900)), "s2 x": "".join(rng.choice(list("ACGTNacgt"), size=3001))}
    fa = tmp_path / "in.fa"
    fa.write_text("".join(">%s\n%s\n" % kv for kv in seqs.items()))
    out = tmp_path / "orfs.fa"
    gt.dna2orfs(str(fa), str(out), from_atg=from_atg, longest=longest, genetic_code="5")
    got = _records(out.read_text())
    lib = gencode.library(5)
    import py2dict
    want = []
    for name in py2dict.py2_order(list(seqs)):
        if longest:
            want.append((name + "_longestORF", ref.get_orfs(seqs[name], lib, longest=True)))
        else:
            want += [(None, o) for o in ref.get_orfs(seqs[name], lib, from_atg=from_atg)]
    if longest:
        assert got == want
    else:
        assert [b for _, b in got] == [b for _, b in want]


def test_sharded_run_table_with_code(mg):
    from magot_b200 import engine, gencode, _lib
    n = _lib.device_count()
    if n < 2:
        pytest.skip("needs at least two CUDA devices")
    rng = np.random.default_rng(3)
    contigs, segs = _random_plan_case(rng)
    tbl, names = _table(segs, True)
    reps = []
    for d in range(n):
        h = engine.DeviceGenome([a.size for a in contigs], device=d)
        for i, a in enumerate(contigs):
            h.pack(i, a)
        h.finalize()
        reps.append(h)
    sh = engine.ShardedGenome(reps)
    t5 = gencode.codon64(5)
    assert sh.run_table(tbl, protein=True, codon64=t5)[0] == engine.run_table(reps[0], tbl, protein=True, codon64=t5)[0]
    sh.close()
