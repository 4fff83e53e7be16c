#!/usr/bin/env python3
"""Generates the committed golden fixtures in tests/golden/ by running the REFERENCE's own
code (shimmed for Python 3 by oracle/make_ref.py, Python-2.7 dict order restored by
oracle/ref_runner.py).  Run in the build container, where /root/reference exists:

    python tests/golden/make_golden.py

Writes
  ref_test_data/*.gz   the reference's data fixtures (test_data/, DATA not source), gzipped,
                       so the GPU box -- which has no /root/reference -- can run the same cases
  manifest.json        POSIX cksum + byte count of the reference's stdout for every whole-file
                       case (plus the three cksums hard-coded in test_data/test_suite.py)
  obiroi_gff2fasta_protein.fa.gz
                       the whole stdout of gff2fasta seq_type=protein on the O.biroi pair, gzipped
  kat.json             known-answer vectors for Sequence.reverse_compliment / translate /
                       get_orfs / BaseAnnotation.get_seq clamping produced by the reference
"""
import gzip
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_runner            # noqa: E402
import surrogate_c14         # noqa: E402
from cksum import cksum      # noqa: E402

REF_DATA = "/root/reference/test_data"
DATA_FILES = ["O.biroi_refseqGenomeSubset.fasta", "O.biroi_NCBIrefseq_gff3Subset.gff", "StandardGTF.gtf",
              "transcriptlessGTF.gtf", "minimalGFF3.gff", "CDSannotations.cds"]


def copy_data():
    out = os.path.join(HERE, "ref_test_data")
    os.makedirs(out, exist_ok=True)
    for f in DATA_FILES:
        with open(os.path.join(REF_DATA, f), "rb") as fh:
            raw = fh.read()
        with open(os.path.join(out, f + ".gz"), "wb") as fh:
            fh.write(gzip.compress(raw, 9, mtime=0))


def whole_file_cases(tmp):
    g = ref_runner.ref()
    T = REF_DATA + "/"
    ob_fa, ob_gff = T + DATA_FILES[0], T + DATA_FILES[1]
    c14 = os.path.join(tmp, "C14.fasta")
    with open(c14, "w", encoding="latin-1", newline="\n") as fh:
        fh.write(surrogate_c14.build(T + "StandardGTF.gtf", T + "CDSannotations.cds"))
    cases = {}

    def put(name, text):
        c, n = cksum(text)
        cases[name] = {"cksum": c, "bytes": n}

    # --- hard-coded by the reference's own test-suite (test_data/test_suite.py:8,12-14)
    cases["suite:exclude_from_fasta"] = {"cksum": 1797510917, "bytes": 256187}
    cases["suite:gff2fasta_C14_StandardGTF"] = {"cksum": 2836090577, "bytes": 690750}
    cases["suite:gff2fasta_C14_StandardGTF_protein"] = {"cksum": 111942461, "bytes": 233762}
    cases["suite:cds2pep"] = {"cksum": 111942461, "bytes": 233762}

    # --- BASELINE config 1: O.biroi FASTA + GFF3
    put("obiroi:gff2fasta", ref_runner.gff2fasta(ob_fa, ob_gff))
    prot = ref_runner.gff2fasta(ob_fa, ob_gff, seq_type="protein")
    put("obiroi:gff2fasta_protein", prot)
    with open(os.path.join(HERE, "obiroi_gff2fasta_protein.fa.gz"), "wb") as fh:
        fh.write(gzip.compress(prot.encode("latin-1"), 9, mtime=0))
    put("obiroi:gff2fasta_from_exons", ref_runner.gff2fasta(ob_fa, ob_gff, from_exons="True"))
    my = ref_runner.load_genome(ob_fa, ob_gff, base_features=['exon', 'match_part', 'similarity', 'region'],
                                features_to_ignore=['CDS'])
    put("obiroi:exon_transcripts", my.annotations.get_fasta('gene') + "\n")
    my = ref_runner.load_genome(ob_fa, ob_gff)
    put("obiroi:get_fasta_mRNA", my.annotations.get_fasta('mRNA') + "\n")
    put("obiroi:get_fasta_mRNA_protein", my.annotations.get_fasta('mRNA', seq_type="protein") + "\n")
    put("obiroi:mRNA_name_from_Name",
        "\n".join(my.annotations.mRNA[k].get_fasta(name_from='Name') for k in my.annotations.mRNA) + "\n")
    put("obiroi:mRNA_genomic",
        "\n".join(my.annotations.mRNA[k].get_fasta(genomic=True) for k in my.annotations.mRNA) + "\n")
    put("obiroi:genome_fasta", my.get_genome_fasta() + "\n")
    put("obiroi:cds_get_seq",
        "\n".join(k + "\t" + my.annotations.CDS[k].get_seq() for k in my.annotations.CDS) + "\n")

    # --- BASELINE config 2: surrogate C14 x three annotation formats
    for gff in ("StandardGTF.gtf", "transcriptlessGTF.gtf", "minimalGFF3.gff"):
        put("c14:%s" % gff, ref_runner.gff2fasta(c14, T + gff))
        put("c14:%s:protein" % gff, ref_runner.gff2fasta(c14, T + gff, seq_type="protein"))
    put("c14:StandardGTF.gtf:genomic", ref_runner.gff2fasta(c14, T + "StandardGTF.gtf", genomic="True"))
    put("c14:StandardGTF.gtf:longest", ref_runner.gff2fasta(c14, T + "StandardGTF.gtf", longest="True"))
    my = ref_runner.load_genome(c14, T + "StandardGTF.gtf")
    put("c14:StandardGTF.gtf:get_fasta_transcript", my.annotations.get_fasta('transcript') + "\n")
    return cases


def aligner_inputs():
    """Synthetic blast -outfmt 10 and exonerate outputs against the O.biroi contigs (committed: aligner_inputs/)."""
    rnd = random.Random(424242)
    contigs = []
    name = None
    with open(os.path.join(REF_DATA, DATA_FILES[0])) as fh:
        for line in fh:
            if line.startswith(">"):
                name = line[1:].strip()
                contigs.append([name, 0])
            else:
                contigs[-1][1] += len(line.strip())
    out = os.path.join(HERE, "aligner_inputs")
    os.makedirs(out, exist_ok=True)
    # blast: qseqid,sseqid,pident,length,mismatch,gapopen,qstart,qend,sstart,send,evalue,bitscore
    rows = []
    for i in range(70):
        full, L = rnd.choice(contigs)
        q = "query%02d" % rnd.randrange(25)              # repeated query ids -> ID-1, ID-2 ...
        n = rnd.randrange(30, min(1500, L // 2))
        a = rnd.randrange(1, L - n)
        s0, s1 = (a, a + n) if rnd.random() < 0.5 else (a + n, a)
        rows.append(",".join([q, full.split()[0], "%.2f" % rnd.uniform(70, 100), str(n), "3", "1", "1", str(n), str(s0), str(s1),
                              "1e-%d" % rnd.randrange(5, 90), "%.1f" % rnd.uniform(50, 900)]))
    rows.insert(10, "short,line,only")                   # fewer than 9 fields: skipped
    rows.append(",".join(["edge", contigs[0][0].split()[0], "99.0", "50", "0", "0", "1", "50", str(contigs[0][1] - 20),
                          str(contigs[0][1] + 30), "0.0", "99"]))          # runs off the contig end: slice clamps
    with open(os.path.join(out, "obiroi_blast.csv"), "w") as fh:
        fh.write("\n".join(rows) + "\n")
    # exonerate: Query / Target header lines + vulgar line (label, query length, target length triples)
    blocks = []
    big = [c for c in contigs if c[1] > 80000]
    for i in range(40):
        full, L = rnd.choice(big)
        q = "prot%02d some description" % rnd.randrange(28)   # repeats against the same target -> numbered
        plus = rnd.random() < 0.5
        pos = rnd.randrange(5000, L - 60000)
        triples = []
        span = 0
        nex = rnd.randrange(1, 7)
        for e in range(nex):
            m = 3 * rnd.randrange(10, 150)
            triples += ["M", str(m // 3), str(m)]
            span += m
            if rnd.random() < 0.3:
                triples += ["G", "0", "3", "M", "20", "60"]
                span += 63
            if rnd.random() < 0.15:
                triples += ["F", "0", "1", "M", "5", "15"]
                span += 16
            if e != nex - 1:
                if rnd.random() < 0.5:
                    triples += ["S", "0", "2"]
                    span += 2
                intron = rnd.randrange(60, 4000)
                triples += ["5", "0", "2", "I", "0", str(intron), "3", "0", "2"]
                span += intron + 4
                if rnd.random() < 0.5:
                    triples += ["S", "1", "1"]
                    span += 1
        ts, te = (pos, pos + span) if plus else (pos + span, pos)
        target = full + (":[revcomp]" if not plus and rnd.random() < 0.5 else ("[revcomp]" if not plus else ""))
        blocks.append("C4 Alignment:\n------------\n         Query: %s\n        Target: %s\n         Model: protein2genome:local\n"
                      "     Raw score: %d\n\nvulgar: %s 0 %d . %s %d %d %s %d %s\n" %
                      (q, target, rnd.randrange(100, 2000), q.split()[0], span // 3, full.split()[0], ts, te, "+" if plus else "-",
                       rnd.randrange(100, 2000), " ".join(triples)))
    with open(os.path.join(out, "obiroi_exonerate.txt"), "w") as fh:
        fh.write("Command line: [exonerate --model protein2genome q.fa t.fa --showvulgar yes]\n\n" + "\n".join(blocks) +
                 "-- completed exonerate analysis\n")
    return os.path.join(out, "obiroi_blast.csv"), os.path.join(out, "obiroi_exonerate.txt")


def aligner_cases(cases):
    blast, exo = aligner_inputs()
    ob_fa = os.path.join(REF_DATA, DATA_FILES[0])
    for name, text in (("obiroi:blast_csv2fasta", ref_runner.blast_csv2fasta(ob_fa, blast)),
                       ("obiroi:exonerate2fasta", ref_runner.exonerate2fasta(ob_fa, exo))):
        c, n = cksum(text)
        cases[name] = {"cksum": c, "bytes": n}
    model = {"blast": ref_runner.aligner_model(ob_fa, "read_blast_csv", blast),
             "exonerate": ref_runner.aligner_model(ob_fa, "read_exonerate", exo)}
    with open(os.path.join(HERE, "aligner_model.json"), "w") as fh:
        json.dump(model, fh, indent=0)


def mask_inputs():
    """Small FASTA + GFF for mask_from_gff (committed under aligner_inputs/): soft-masked and IUPAC bases, bytes outside
    the packed alphabet, a repeated header, CRLF lines, overlapping / duplicate / clamped / empty intervals."""
    rnd = random.Random(99)
    out = os.path.join(HERE, "aligner_inputs")
    os.makedirs(out, exist_ok=True)
    alpha = "ACGT" * 8 + "acgt" * 6 + "NNnn" + "RYKMrykmSWBDHVswbdhv*-. x"
    seqs = [("ctgA desc one", 5000), ("ctgB", 1234), ("ctgC\tTabbed", 801), ("ctgA second copy replaces the first", 3000),
            ("short", 7), ("ctgD", 40000)]
    with open(os.path.join(out, "mask.fasta"), "w", newline="") as fh:
        for name, n in seqs:
            s = "".join(rnd.choice(alpha) for _ in range(n))
            fh.write(">" + name + "\n")
            eol = "\r\n" if name == "ctgB" else "\n"
            for k in range(0, n, 70):
                fh.write(s[k:k + 70] + eol)
    lens = {"ctgA": 3000, "ctgB": 1234, "ctgC": 801, "short": 7, "ctgD": 40000}
    rows = ["##gff-version 3"]
    for i in range(300):
        c = rnd.choice(list(lens))
        L = lens[c]
        a = rnd.randrange(1, L + 1)
        b = min(L, a + rnd.randrange(0, 400))
        ftype = rnd.choice(["CDS", "CDS", "CDS", "exon", "gene"])
        rows.append("\t".join([c, "src", ftype, str(a), str(b), ".", rnd.choice("+-"), ".", "ID=f%d" % i]))
    rows.append("\t".join(["ctgA", "src", "CDS", "10", "20", ".", "+", ".", "ID=dup"]))
    rows.append("\t".join(["ctgA", "src", "CDS", "10", "20", ".", "+", ".", "ID=dup"]))
    rows.append("\t".join(["ctgA", "src", "CDS", "15", "12", ".", "+", ".", "ID=backwards"]))          # empty slice
    rows.append("\t".join(["ctgB", "src", "CDS", "1", "1234", ".", "+"]))                               # 6 tabs only: still counts
    rows.append("ctgB\tsrc\tCDS\t5\t9")                                                               # 4 tabs: ignored
    with open(os.path.join(out, "mask.gff"), "w") as fh:
        fh.write("\n".join(rows) + "\n")
    soft_extra = list(rows)
    soft_extra.append("\t".join(["short", "src", "CDS", "3", "500", ".", "+", ".", "ID=clamped"]))        # soft: slice clamps
    soft_extra.append("\t".join(["ctgC", "src", "CDS", "0", "5", ".", "+", ".", "ID=zero"]))             # [-1:5] -> empty
    soft_extra.append("\t".join(["ctgC", "src", "CDS", "-20", "-3", ".", "+", ".", "ID=negative"]))       # negative indices
    with open(os.path.join(out, "mask_soft.gff"), "w") as fh:
        fh.write("\n".join(soft_extra) + "\n")
    return os.path.join(out, "mask.fasta"), os.path.join(out, "mask.gff"), os.path.join(out, "mask_soft.gff")


def mask_cases(cases):
    fa, gff, gff_soft = mask_inputs()
    ob_fa, ob_gff = os.path.join(REF_DATA, DATA_FILES[0]), os.path.join(REF_DATA, DATA_FILES[1])
    runs = {"mask:soft": (fa, gff_soft, {}),
            "mask:soft_keep_case": (fa, gff_soft, {"overwrite_softmask": "False"}),
            "mask:hard": (fa, gff, {"mask_type": "hard"}),
            "mask:hard_keep_case_exon": (fa, gff, {"mask_type": "hard", "overwrite_softmask": "F", "feature_type": "exon"}),
            "mask:obiroi_soft": (ob_fa, ob_gff, {}),
            "mask:obiroi_hard_exon": (ob_fa, ob_gff, {"mask_type": "hard", "feature_type": "exon", "overwrite_softmask": "False"})}
    for name, (a, b, kw) in runs.items():
        c, n = cksum(ref_runner.mask_from_gff(a, b, **kw))
        cases[name] = {"cksum": c, "bytes": n}


ALPHABETS = {
    "acgt": "ACGT",
    "mixed": "ACGTacgtNn",
    "iupac": "ACGTacgtNnRYKMSWBDHVrykm-*. xU",
}


GFF_FORMATS = ["simple gff3", "extended gff3", "exon added gff3", "gtf", "augustus hint CDS b2h 4", "augustus hint CDSpart M"]
AUGUSTUS_PRESET = dict(features_to_ignore=['gene', 'transcript', 'stop_codon', 'terminal', 'internal', 'initial', 'intron',
                                           'start_codon', 'single'],
                       parent_field=None, parents_hierarchy=['transcript_id', 'gene_id'], IDfield=None)


def gff_writer_cases(cases):
    """SURVEY 8(f)-4: write_gff / get_gff / convert_gff (genome.py:228-238, :616-645, :733-778; genome_tools.py:527-545).
    A case the reference crashes on is recorded as {"raises": <exception name>}."""
    T = REF_DATA + "/"
    # hard-coded by the reference's own test-suite (test_data/test_suite.py:15-17)
    cases["suite:convert_gff_minimalGFF3_gff3_gtf"] = {"cksum": 1904390924, "bytes": 226225}
    cases["suite:convert_gff_StandardGTF_gtf_gff3"] = {"cksum": 2934568300, "bytes": 276674}
    cases["suite:convert_gff_StandardGTF_gtf_exon_added_gff3"] = {"cksum": 2624776569, "bytes": 512324}

    def put(name, fn):
        try:
            c, n = cksum(fn())
            cases[name] = {"cksum": c, "bytes": n}
        except Exception as e:            # noqa: BLE001 -- the reference's own crash is the expected behaviour
            cases[name] = {"raises": type(e).__name__}

    for f in ("StandardGTF.gtf", "minimalGFF3.gff", "transcriptlessGTF.gtf", "O.biroi_NCBIrefseq_gff3Subset.gff"):
        for fmt in GFF_FORMATS:
            put("gffwrite:%s:%s" % (f, fmt), lambda: ref_runner.write_gff(T + f, fmt))
    ob = T + "O.biroi_NCBIrefseq_gff3Subset.gff"
    for fmt in ("simple gff3", "extended gff3"):
        put("gffwrite:obiroi_exon_based:%s" % fmt,
            lambda: ref_runner.write_gff(ob, fmt, base_features=['exon', 'match_part', 'similarity', 'region'],
                                         features_to_ignore=['CDS']))
    # presets='augustus' is an exec() of these assignments (genome.py:262-268); the shim cannot rebind locals under
    # Python 3, so the reference is run with the same values passed explicitly
    for fmt in ("simple gff3", "gtf"):
        put("gffwrite:StandardGTF.gtf:augustus_preset:%s" % fmt,
            lambda: ref_runner.write_gff(T + "StandardGTF.gtf", fmt, **AUGUSTUS_PRESET))


def position_dic_cases():
    """position_dic (genome.py:981-1100) run by the reference on a small genome: at_content, fill / count from
    annotations, sliding_window_calculate (sum / average -> dict, annotation_set with its region-merging quirks, verbose
    output).  Inputs travel inside the fixture.  Python-2.7 orders are restored where a dict is iterated."""
    import contextlib
    import io
    import numpy
    from py2dict import py2_order
    g = ref_runner.ref()
    rnd = random.Random(4242)

    def contig(n, at):
        out = []
        while len(out) < n:
            rich = rnd.random() < 0.3
            run = rnd.randint(20, 400)
            p = at if not rich else 0.9
            out.extend(rnd.choice("ATat" if rnd.random() < p else "CGcgNn") for _ in range(run))
        return "".join(out[:n])

    seqs = {"ctgA": contig(5003, 0.5), "ctgB some text": contig(1203, 0.35), "ctgC": contig(64, 0.5), "ctgD": contig(300, 0.2)}
    fasta = "".join(">%s\n%s\n" % (k, "\n".join(v[i:i + 70] for i in range(0, len(v), 70))) for k, v in seqs.items())
    gff_lines = []
    k = 0
    for seqid, L in (("ctgA", 5003), ("ctgB some text", 1203), ("ctgD", 300)):
        for gi in range(3):
            k += 1
            a = rnd.randint(1, L - 200)
            gff_lines.append("%s\tsyn\tgene\t%d\t%d\t.\t+\t.\tID=g%d" % (seqid, a, a + 180, k))
            gff_lines.append("%s\tsyn\tmRNA\t%d\t%d\t.\t+\t.\tID=t%d;Parent=g%d" % (seqid, a, a + 180, k, k))
            gff_lines.append("%s\tsyn\tCDS\t%d\t%d\t.\t+\t0\tID=c%da;Parent=t%d" % (seqid, a, a + 60, k, k))
            gff_lines.append("%s\tsyn\tCDS\t%d\t%d\t.\t+\t0\tID=c%db;Parent=t%d" % (seqid, a + 100, a + 180, k, k))
    gff = "\n".join(gff_lines) + "\n"

    def fresh(dtype=bool):
        gs = g.GenomeSequence(fasta)
        ref_runner.reorder_genome_sequence(gs)
        pd = g.position_dic(gs, dtype=dtype)
        items = {kk: pd[kk] for kk in py2_order(list(pd))}       # a position_dic is a py2 dict itself
        pd.clear()
        pd.update(items)
        return gs, pd

    aset = g.read_gff(gff)
    ref_runner.reorder_annotation_set(aset)
    out = {"fasta": fasta, "gff": gff, "order": None, "at_content": {}, "fill": {}, "count": {}, "windows": []}
    gs, pd = fresh()
    out["order"] = list(pd)
    pd.at_content(gs)
    out["at_content"] = {kk: "".join("1" if x else "0" for x in v) for kk, v in pd.items()}
    at_pd = pd
    for feature, fill_type in (("CDS", "coords"), ("gene", "coords"), ("CDS", "start")):
        _, pd = fresh()
        pd.fill_from_annotations(aset, feature, fill_type=fill_type)
        out["fill"]["%s:%s" % (feature, fill_type)] = {kk: "".join("1" if x else "0" for x in v) for kk, v in pd.items()}
    _, pd = fresh(dtype=int)
    pd.fill_from_annotations(aset, "CDS", fill_with="coords[0] % 3")
    out["fill"]["CDS:coords:int:coords[0] % 3"] = {kk: [int(x) for x in v] for kk, v in pd.items()}
    _, pd = fresh()
    pd.fill_from_annotations(aset, "CDS")
    out["count"]["gene_over_CDS_fill"] = pd.count_from_annotations(aset, "gene")
    out["count"]["mRNA_over_at"] = at_pd.count_from_annotations(aset, "mRNA")
    for (w, j, op, output, thr, excl) in [(50, 1, "sum", "dict", 1, []), (100, 25, "sum", "dict", 1, []),
                                          (64, 64, "average", "dict", 1, ["ctgD"]), (7, 3, "sum", "dict", 1, []),
                                          (63, 1, "sum", "dict", 1, []), (64, 1, "sum", "dict", 1, []),
                                          (50, 1, "sum", "annotation_set", 40, []), (50, 10, "sum", "annotation_set", 35, []),
                                          (40, 5, "average", "annotation_set", 0.8, []), (30, 7, "sum", "annotation_set", 0, []),
                                          (100, 1, "sum", "annotation_set", 101, []), (20, 20, "sum", "annotation_set", 12, ["ctgA"])]:
        for verbose in (False, True):
            g.verbose = verbose
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf):
                r = at_pd.sliding_window_calculate(w, window_jump=j, operation=op, output=output, threshold=thr, seqs_to_exclude=excl)
            g.verbose = True
            if output == "dict":
                res = {kk: [float(x) if op == "average" else int(x) for x in v] for kk, v in r.items()}
                key_order = py2_order(list(r))
            else:
                ref_runner.reorder_annotation_set(r)
                res = [[kk, list(v.coords), v.seqid] for kk, v in r.region.items()]
                key_order = None
            if verbose and output == "annotation_set":
                continue            # the reference prints the regions in the order of a py2 dict the shim cannot replay
            out["windows"].append({"window": w, "jump": j, "operation": op, "output": output, "threshold": thr, "exclude": excl,
                                   "verbose": verbose, "result": res, "key_order": key_order, "stdout": buf.getvalue()})
    return out


def library_vectors():
    """Sequence.translate(library=...) (genome.py:795, :814-817) with caller-supplied codon dicts, run by the reference:
    the vertebrate mitochondrial code, a library with only three entries (everything else -> 'X'), and one whose extra
    keys can never match an upper-cased triplet (lower case, wrong length)."""
    g = ref_runner.ref()
    rnd = random.Random(77)
    std = dict(zip([a + b + c for a in "TCAG" for b in "TCAG" for c in "TCAG"],
                   "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"))
    mito = dict(std, AGA="*", AGG="*", ATA="M", TGA="W")
    sparse = {"ATG": "m", "TAA": "#", "GGG": "X"}
    odd = dict(std, atg="?", AT="?", ATGA="?", TTT="f")
    libs = {"mito": mito, "sparse": sparse, "odd_keys": odd}
    seqs = ["", "AT", "ATG", "ATGA", "NNNATGAGATAA", "atgagaTGAata", "TTTtttTTNAGG"]
    for alpha in ("ACGT", "ACGTacgtNn-RY"):
        for n in (3, 7, 32, 100, 999):
            seqs.append("".join(rnd.choice(alpha) for _ in range(n)))
    out = {"libraries": libs, "vectors": []}
    for lname, lib in libs.items():
        for s in seqs:
            for frame in (0, 1, 2):
                for strand in "+-":
                    for trimX in (True, False):
                        try:
                            r = g.Sequence(s).translate(library=lib, frame=frame, strand=strand, trimX=trimX)
                        except IndexError:
                            r = "!IndexError"
                        out["vectors"].append([lname, s, frame, strand, trimX, r])
    return out


def kat_vectors():
    g = ref_runner.ref()
    rnd = random.Random(20261018)
    vec = {"reverse_compliment": [], "translate": [], "get_orfs": [], "get_seq": []}
    seqs = ["", "A", "AC", "ACG", "ACGT", "NNNATG", "acgRYKn-", "ATGTAA", "atgtaa", "ATGNNNTAA", "TAATAGTGA",
            "ATG-AATAG", "NNATGAAATAG", "XATGCC"]
    for name, alpha in ALPHABETS.items():
        for n in (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 31, 32, 33, 63, 64, 65, 100, 257, 1000):
            seqs.append("".join(rnd.choice(alpha) for _ in range(n)))
    for s in seqs:
        vec["reverse_compliment"].append([s, str(g.Sequence(s).reverse_compliment())])
        for frame in (0, 1, 2):
            for strand in "+-":
                for trimX in (True, False):
                    try:
                        r = g.Sequence(s).translate(frame=frame, strand=strand, trimX=trimX)
                    except IndexError:
                        r = "!IndexError"
                    vec["translate"].append([s, frame, strand, trimX, r])
    orf_inputs = [s for s in seqs if len(s) >= 3]
    for n in (300, 999, 2000):
        # stop-poor sequence so that long ORFs exist
        orf_inputs.append("".join(rnd.choice("ACG" * 6 + "T" + "Nn") for _ in range(n)))
    for s in orf_inputs:
        for from_atg in (False, True):
            vec["get_orfs"].append([s, from_atg, g.Sequence(s).get_orfs(from_atg=from_atg)])
        try:
            lo = g.Sequence(s).get_orfs(longest=True)
        except IndexError:
            lo = "!IndexError"
        vec["get_orfs"].append([s, "longest", lo])
    # BaseAnnotation.get_seq: Python-slice clamping at contig ends (genome.py:603-608)
    contig = "".join(rnd.choice("ACGTacgtN") for _ in range(50))
    gs = g.GenomeSequence(">c1\n" + contig + "\n")
    for (a, b) in [(1, 50), (1, 1), (50, 50), (10, 20), (45, 60), (50, 80), (51, 60), (0, 5), (0, 50), (0, 60),
                   (-3, 10), (-3, 60), (30, 29), (7, 7)]:
        for strand in "+-.":
            aset = g.AnnotationSet()
            my = g.Genome(gs)
            my.annotations = aset
            aset.genome = my
            base = g.BaseAnnotation("x", "c1", tuple(sorted((a, b))), "CDS", None, strand, {}, aset)
            vec["get_seq"].append([contig, a, b, strand, str(base.get_seq())])
    return vec


def main():
    import tempfile
    if "--only-position-dic" in sys.argv:
        with open(os.path.join(HERE, "position_dic.json"), "w") as fh:
            json.dump(position_dic_cases(), fh, indent=0)
        print("wrote position_dic.json")
        return
    if "--only-library-kat" in sys.argv:      # add the custom-codon-table vectors to the existing kat.json
        with open(os.path.join(HERE, "kat.json")) as fh:
            kat = json.load(fh)
        kat["translate_library"] = library_vectors()
        with open(os.path.join(HERE, "kat.json"), "w") as fh:
            json.dump(kat, fh, indent=0)
        print("kat.json: +", len(kat["translate_library"]["vectors"]), "library vectors")
        return
    if "--only-gff-writers" in sys.argv:      # add the writer cases to the existing manifest
        with open(os.path.join(HERE, "manifest.json")) as fh:
            cases = json.load(fh)
        gff_writer_cases(cases)
        with open(os.path.join(HERE, "manifest.json"), "w") as fh:
            json.dump(cases, fh, indent=1, sort_keys=True)
        print("manifest now holds", len(cases), "whole-file cases")
        return
    copy_data()
    with tempfile.TemporaryDirectory() as tmp:
        cases = whole_file_cases(tmp)
    aligner_cases(cases)
    mask_cases(cases)
    gff_writer_cases(cases)
    with open(os.path.join(HERE, "manifest.json"), "w") as fh:
        json.dump(cases, fh, indent=1, sort_keys=True)
    with open(os.path.join(HERE, "kat.json"), "w") as fh:
        kat = kat_vectors()
        kat["translate_library"] = library_vectors()
        json.dump(kat, fh, indent=0)
    with open(os.path.join(HERE, "position_dic.json"), "w") as fh:
        json.dump(position_dic_cases(), fh, indent=0)
    print("wrote", len(cases), "whole-file cases")


if __name__ == "__main__":
    main()
