#!/usr/bin/env python3
"""Drop-in mirror of the sequence entry points of MAGOT's `genome_tools` script
(reference: /root/reference/genome_tools.py).

Usage is unchanged:  python -m magot_b200.genome_tools <function> [positional ...] [key=value ...]
Every argument arrives as a string ("True"/"False" are interpreted inside the tools, as in the
reference) and every tool prints to stdout exactly what the reference prints.

Kept (file:line in genome_tools.py): gff2fasta :324, cds2pep :664, coords2fasta :656,
get_seq_from_fasta :483, exclude_from_fasta :377, extract_upstream_downstream :457,
blast_csv2fasta :265, exonerate2fasta :274, mask_from_gff :394, convert_gff :527,
dna2orfs :145 (the reference's version cannot run -- it calls str.translate with keyword
arguments -- this one does what it intended, on the device).  New: call_orfs, start-to-stop
ORF calling with genome coordinates (GFF3, protein or CDS nucleotide output), check_cds, a gene-model check (start /
stop codons, in-frame stops, frame, splice sites, codon usage), and predict_cds, the longest ORF of each exon-only transcript
model as GFF3 CDS rows, protein or CDS text.  The dispatcher (main :25-45)
keeps the grammar but looks the function up in a table instead of eval()-ing a string.
"""
import sys

import numpy as np

from . import genome
from . import engine
from . import gencode


def _truth(s):
    """eval("True") / eval("False") of the reference, without eval."""
    if s in ("True", "False"):
        return s == "True"
    if isinstance(s, bool):
        return s
    raise NameError("name %r is not defined" % (s,))


def gff2fasta(genome_sequence, gff, from_exons="False", seq_type="nucleotide", longest="False", genomic="False",
              genetic_code="1"):
    """genome_tools.py:324-330.  genetic_code=<NCBI table id> (new; default 1, the reference's table) translates
    seq_type=protein, e.g. genetic_code=5 for insect mitochondria."""
    code = gencode.check(genetic_code)
    my_genome = genome.Genome(genome_sequence)
    if from_exons == "True":
        # the reference passes features_to_ignore as the *string* "CDS" (substring test) after renaming
        # exon -> CDS, so every exon and CDS line is ignored; reproduced as is.
        my_genome.read_gff(gff, features_to_ignore="CDS", features_to_replace=[('exon', 'CDS')])
    else:
        my_genome.read_gff(gff)
    print(my_genome.annotations.get_fasta('gene', seq_type=seq_type, longest=_truth(longest), genomic=_truth(genomic),
                                          genetic_code=code))


def convert_gff(gff, input_format, output_format):
    """genome_tools.py:527-545 -- re-write an annotation file: input `gff3` or a read_gff preset name (anything else, e.g.
    `gtf`, reads with the defaults), output `gff3`, `gtf` or `exon_added_gff3`.  Host-only (no sequence is touched)."""
    presets = None if input_format == 'gff3' else input_format
    if output_format == 'gff3':
        gff_format = "simple gff3"
    elif output_format == 'gtf':
        gff_format = 'gtf'
    elif output_format == "exon_added_gff3":
        gff_format = "exon added gff3"
    else:
        print("currently only writes 'gff3' and 'gtf' format")
        return None
    annotations = genome.read_gff(gff, presets=presets)
    print(genome.write_gff(annotations, gff_format))


def blast_csv2fasta(genome_sequence, blast_csv):
    """genome_tools.py:265-271 -- one record per blast hit (`match`), all hits through ONE device plan."""
    my_genome = genome.Genome(genome_sequence)
    my_genome.read_blast_csv(blast_csv)
    print(my_genome.annotations.get_fasta('match'))


def exonerate2fasta(genome_sequence, exonerate_file):
    """genome_tools.py:274-280 -- one record per exonerate alignment (`match`), its match_parts spliced."""
    my_genome = genome.Genome(genome_sequence)
    my_genome.read_exonerate(exonerate_file)
    print(my_genome.annotations.get_fasta('match'))


def mask_from_gff(genome_sequence, gff, mask_type="soft", overwrite_softmask="True", feature_type="CDS"):
    """genome_tools.py:394-428 -- soft- (lower-case) or hard- ('N') mask every `feature_type` interval of a GFF and print
    the genome, one line per sequence.  The intervals are scattered onto the packed genome on the device (K5).
    Kept from the reference: seqid = first word of the header, a repeated header starts the sequence over, any GFF line with
    more than 5 tabs counts, coordinates follow Python slice rules, the printed order is the reference's dict order.
    Not kept: a hard mask whose slice is clamped changes the sequence LENGTH in the reference (list slice assignment);
    that raises NotImplementedError here."""
    with open(genome_sequence, "rb") as fh:
        data = fh.read()
    if overwrite_softmask in ("True", "T", "true", "t", "TRUE"):
        upper_first = True
    elif overwrite_softmask in ("False", "F", "false", "f", "FALSE"):
        upper_first = False
    else:
        upper_first = None
    seqs = {}
    working = None
    lines = data.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()                                     # no line after the final newline
    for line in lines:
        if line[:1] == b">":
            working = line.decode("latin-1").split()[0][1:].replace('\r', '')
            seqs[working] = []
        elif line or working is None:
            if working is None:
                raise KeyError("")                      # sequence before the first header: genome_dict[""] in the reference
            if upper_first is None:
                print("Invalid option for 'overwrite_softmask', argument accepts 'True' or 'False'")
                return None
            seqs[working].append(line.replace(b"\r", b""))
    names = genome._order(list(seqs))
    arrays = [np.frombuffer(b"".join(seqs[n]), dtype=np.uint8) for n in names]
    index = {n: i for i, n in enumerate(names)}
    cid, lo, hi = [], [], []
    with open(gff, encoding="latin-1", newline="\n") as fh:
        for line in fh:
            if line.count('\t') > 5:
                fields = line.split('\t')
                if fields[2] == feature_type:
                    start, stop = int(fields[3]), int(fields[4])
                    ci = index[fields[0]]                # KeyError for an unknown seqid, as the reference
                    a, b, _ = slice(start - 1, stop).indices(arrays[ci].size)
                    b = max(a, b)
                    if mask_type == "soft":
                        pass
                    elif mask_type == "hard":
                        if b - a != max(1 + stop - start, 0):
                            raise NotImplementedError("hard mask %s:%d-%d is clamped by the sequence end: the reference would "
                                                      "change the sequence length here" % (fields[0], start, stop))
                    else:
                        print("Invalid option for mask_type, argument accepts 'soft' and 'hard'")
                        return None
                    cid.append(ci)
                    lo.append(a)
                    hi.append(b)
    g = engine.DeviceGenome([a.size for a in arrays], device=0)
    try:
        for ci, a in enumerate(arrays):
            g.pack(ci, a)
        g.finalize()
        g.mask(cid, lo, hi, hard=(mask_type == "hard"), upper_first=bool(upper_first))
        for ci, n in enumerate(names):
            L = arrays[ci].size
            print(">" + n + "\n" + (g.fetch(ci, 0, L).decode("latin-1") if L else ""))
    finally:
        g.close()


def cds2pep(fasta_file, genetic_code="1"):
    """genome_tools.py:664-675 -- all records are translated in ONE device launch.  genetic_code=<NCBI table id> (new;
    default 1, the reference's table)."""
    code = gencode.check(genetic_code)
    headers = []
    seqs = []
    working = []
    have = False
    order = []                       # ('h', idx) / ('s', idx) in print order
    with open(fasta_file, encoding="latin-1", newline="\n") as fh:
        for original_line in fh:
            line = original_line.replace('\n', '').replace('\r', '')
            if line[0] == '>':
                if have:
                    seqs.append("".join(working).encode("latin-1"))
                    order.append(('s', len(seqs) - 1))
                    working = []
                    have = False
                headers.append(line)
                order.append(('h', len(headers) - 1))
            else:
                working.append(line)
                if line != "":
                    have = True
    seqs.append("".join(working).encode("latin-1"))
    order.append(('s', len(seqs) - 1))
    peps = genome._translate_many(seqs, library=gencode.library(code) if code != 1 else None)
    out = []
    for kind, idx in order:
        out.append(headers[idx] if kind == 'h' else str(peps[idx]))
    sys.stdout.write("\n".join(out) + "\n")


def coords2fasta(fasta_file, seqid, start, stop, truncate_names="False"):
    """genome_tools.py:656-661: 1-based inclusive coordinates, Python slice clamping."""
    print(">" + seqid + ":" + start + "-" + stop)
    print(genome.Genome(fasta_file, truncate_names=_truth(truncate_names)).genome_sequence[seqid][int(start) - 1:int(stop)])


def get_seq_from_fasta(genome_sequence, seq_name, truncate_names="False"):
    """genome_tools.py:483-485."""
    my_genome = genome.Genome(genome_sequence, truncate_names=_truth(truncate_names))
    print(my_genome.get_scaffold_fasta(seq_name))


def exclude_from_fasta(fasta, exclude_list, just_firstword="False"):
    """genome_tools.py:377-391 (records in the reference's dict order)."""
    my_fasta = genome.Genome(fasta)
    try:
        exlist = open(exclude_list).read().replace('\r', '').split('\n')
    except Exception:
        exlist = exclude_list.split(',')
    for seqid in my_fasta.genome_sequence:
        seqid_fixed = seqid.split()[0] if just_firstword == "True" else seqid
        if seqid_fixed not in exlist:
            print('>' + seqid + '\n' + my_fasta.genome_sequence[seqid])


def extract_upstream_downstream(genome_sequence, gff, sequence_length, stream, feature_type="gene", namefrom="ID",
                                truncate_names="True"):
    """genome_tools.py:457-480.  All flanks are fetched in one device plan; the slice arithmetic
    (including Python's negative-index semantics for flanks that run off the contig start) is the
    device's, via start-1/end == Python slice bounds."""
    sequence_dict = genome.GenomeSequence(genome_sequence, truncate_names=_truth(truncate_names))
    n = int(sequence_length)
    names, segs = [], []
    have_sequence = False
    last_seg = None
    with open(gff, encoding="latin-1", newline="\n") as fh:
        for line in fh:
            if line.count('\t') > 5 and line[0] != "#":
                fields = line.split('\t')
                if fields[2] == feature_type:
                    name = None
                    coords = sorted([int(fields[3]), int(fields[4])])
                    for attribute in fields[-1].split(';'):
                        if namefrom == attribute.split('=')[0]:
                            name = attribute.split('=')[1].replace('\r', '').replace('\n', '')
                    ci = sequence_dict.contig_index(fields[0])
                    if (stream == "up" and fields[6] == "+") or (stream == "down" and fields[6] == "-"):
                        stop = coords[0] - 1
                        last_seg = (ci, stop - n + 1, stop, 0)          # contig[stop-n:stop]
                        have_sequence = True
                    elif (stream == "down" and fields[6] == "+") or (stream == "up" and fields[6] == "-"):
                        start = coords[1]
                        last_seg = (ci, start + 1, start + n, 1)        # rc(contig[start:start+n])
                        have_sequence = True
                    if not have_sequence:
                        raise UnboundLocalError("local variable 'sequence' referenced before assignment")
                    # like the reference, a feature with another strand value re-uses the previous `sequence`
                    names.append(name)                                   # None -> 'seq<kept so far>' below
                    segs.append(last_seg)
    if not names:
        print("")
        return
    R = len(names)
    zero = np.zeros(R, dtype=np.int32)
    tbl = engine.RecordTable(np.arange(R + 1), [s[0] for s in segs], [s[1] for s in segs], [s[2] for s in segs],
                             [s[3] for s in segs], np.zeros(R, dtype=np.int64), zero, zero, np.zeros(0, dtype=np.uint8))
    text, (nuc_len, _) = sequence_dict._engine().run_table(tbl, want_lengths=True)
    off = np.concatenate(([0], np.cumsum(nuc_len)))
    output_seqs = []
    for k in range(R):
        if nuc_len[k] == n:                                              # genome_tools.py:478
            name = names[k] if names[k] is not None else 'seq' + str(len(output_seqs))
            output_seqs.append('>' + name + '\n' + text[off[k]:off[k + 1]].decode("latin-1"))
    print("\n".join(output_seqs))


def dna2orfs(fasta_location, output_file, from_atg=False, longest=False, min_orf="0", genetic_code="1"):
    """What genome_tools.py:145-180 intended (the reference's own version raises TypeError because
    GenomeSequence values are plain str): six-frame translation of every contig, split on stops,
    written as '>{seqid}-pos:{orf_start}' records, or one '>{seqid}_longestORF' record per contig.
    `min_orf` (residues, new) filters short ORFs on the device; "0" reproduces the reference list.
    `genetic_code` (NCBI table id, new; default 1) sets the residues and the stops, e.g. genetic_code=6 for ciliates."""
    code = gencode.check(genetic_code)
    from .orfs import contig_orfs
    dna = genome.Genome(fasta_location)
    gs = dna.genome_sequence
    with open(output_file, 'w', encoding="latin-1", newline="\n") as out:
        for seq in gs:
            L = len(gs[seq])
            recs, aa = contig_orfs(gs, seq, int(min_orf), genetic_code=code)
            candidate = None
            longest_orf_len = 0
            for r, orf in zip(recs, aa):
                strand_plus = not r["minus"]
                frame = int(r["frame"])
                orf_start = (frame if strand_plus else L - frame) + 3 * int(r["start"])
                if from_atg:
                    output_orf = 'M' + ''.join(orf.split('M')[1:])
                else:
                    output_orf = orf
                if longest:
                    if len(output_orf) > longest_orf_len:
                        candidate = '>' + seq + '_longestORF\n' + output_orf + '\n'
                        longest_orf_len = len(output_orf)
                else:
                    out.write('>' + seq + '-pos:' + str(orf_start) + '\n' + output_orf + '\n')
            if longest:
                out.write(candidate)        # TypeError when the contig has no ORF at all (IndexError in the reference)


ORF_FORMATS = ("gff3", "protein", "nucleotide")


def _orf_order(contig_order, recs):
    """Permutation of mg_orfcall records into call_orfs' order: contigs as listed in contig_order, then lo, '+' before '-',
    then phase (stable)."""
    rank = {int(c): i for i, c in enumerate(contig_order)}
    key = np.array([rank[int(c)] for c in recs["contig"]], dtype=np.int64)
    return np.lexsort((recs["phase"], recs["minus"], recs["lo"], key))


def _orf_lines(names, recs, out_format, seqs=None):
    """Output lines of call_orfs for records already in its order.  names[contig] = seqid; seqs[i] = the protein or
    nucleotide text of recs[i] (not read for gff3).  ORF n (1-based) of a contig is <seqid>_orf<n>."""
    lines = ["##gff-version 3"] if out_format == "gff3" else []
    count = {}
    for i, r in enumerate(recs):
        c = int(r["contig"])
        count[c] = count.get(c, 0) + 1
        seqid = names[c]
        oid = "%s_orf%d" % (seqid, count[c])
        strand = "-" if r["minus"] else "+"
        lo, hi = int(r["lo"]), int(r["hi"])
        if out_format == "gff3":
            sc = int(r["start_codon"])
            attrs = "ID=%s;start_codon=%s" % (oid, "ACGT"[sc >> 4] + "ACGT"[(sc >> 2) & 3] + "ACGT"[sc & 3])
            if int(r["flags"]) & 1:
                attrs += ";partial=3prime"
            lines.append("\t".join((seqid, "magot_b200", "ORF", str(lo + 1), str(hi), ".", strand, ".", attrs)))
        else:
            lines.append(">%s %s:%d-%d(%s)" % (oid, seqid, lo + 1, hi, strand))
            lines.append(seqs[i])
    return lines


def call_orfs(fasta, min_orf="100", genetic_code="1", start_codons="ATG", partial="False", out_format="gff3"):
    """Start-to-stop ORFs of every contig (new; NCBI ORFfinder / EMBOSS getorf style): both strands, the three true phases,
    from the first start codon of each stop-bounded stretch through the stop, at least `min_orf` residues (M included, stop
    excluded).  start_codons: comma-separated codons (default ATG); partial=True adds ORFs that run off the contig end
    without a stop (partial=3prime).  out_format: gff3 (1-based inclusive coordinates), protein (first residue M) or
    nucleotide (start through stop codon, reverse-complemented on '-').  Contigs in the order dna2orfs visits them; within a
    contig by start coordinate, '+' before '-', then phase; IDs <seqid>_orf<n>."""
    from . import orfs
    code = gencode.check(genetic_code)
    if out_format not in ORF_FORMATS:
        raise ValueError("out_format %r is not one of %s" % (out_format, ", ".join(ORF_FORMATS)))
    codons = start_codons.split(",") if isinstance(start_codons, str) else list(start_codons)
    gencode.start64(codons, code)                            # ValueError before any device work
    gs = genome.Genome(fasta).genome_sequence
    order = [gs.contig_index(seq) for seq in gs]
    names = {ci: seq for ci, seq in zip(order, gs)}
    recs, aa = orfs.call_orfs(gs._engine().primary, order, int(min_orf), genetic_code=code, start_codons=codons,
                              partial=_truth(partial))
    recs = recs[_orf_order(order, recs)]
    seqs = None
    if out_format == "protein":
        text = aa.decode("latin-1")
        seqs = [text[int(r["aa_off"]):int(r["aa_off"]) + int(r["len"])] for r in recs]
    elif out_format == "nucleotide" and recs.size:
        R = recs.size
        zero = np.zeros(R, dtype=np.int32)
        tbl = engine.RecordTable(np.arange(R + 1), recs["contig"].astype(np.int32), recs["lo"] + 1, recs["hi"],
                                 recs["minus"].astype(np.int8), np.zeros(R, dtype=np.int64), zero, zero, np.zeros(0, dtype=np.uint8))
        text, (nuc_len, _) = gs._engine().run_table(tbl, want_lengths=True)
        off = np.concatenate(([0], np.cumsum(nuc_len)))
        seqs = [text[off[k]:off[k + 1]].decode("latin-1") for k in range(R)]
    lines = _orf_lines(names, recs, out_format, seqs)
    sys.stdout.write("\n".join(lines) + "\n" if lines else "")


CHECK_FORMATS = ("tsv", "codon_usage")
CHECK_HEADER = "\t".join(("#ID", "nuc_len", "codons", "skip", "rem", "start", "stop", "internal_stops", "first_internal_stop",
                          "ambiguous", "gc", "gc3", "junctions", "noncanonical", "status"))
CODON_USAGE_HEADER = "\t".join(("#codon", "residue", "count", "per_thousand", "fraction"))


def _codon_text(idx):
    """Codon 16*b0 + 4*b1 + b2 (A=0 C=1 G=2 T=3) as text; '.' for 0xFF (absent or ambiguous)."""
    idx = int(idx)
    return "." if idx == 0xFF else "ACGT"[idx >> 4] + "ACGT"[(idx >> 2) & 3] + "ACGT"[idx & 3]


def _check_status(flags):
    """'ok', or the names of the set MG_CHK_* bits joined by commas, in bit order."""
    flags = int(flags)
    names = [n for k, n in enumerate(engine._lib.CHK_FLAGS) if flags >> k & 1]
    return ",".join(names) if names else "ok"


def _check_tsv_lines(names, recs):
    """check_cds out_format=tsv: the header, then one line per record (engine.CHECK_DTYPE) with the columns of CHECK_HEADER.
    internal_stops = n_stop less the terminal stop; first_internal_stop is the codon index of the first stop when there is an
    internal one, else '.'; gc = G/C bases over the bases of unambiguous codons, gc3 = G/C third bases over unambiguous codons,
    both with 4 decimals ('.' without an unambiguous codon)."""
    lines = [CHECK_HEADER]
    for name, r in zip(names, recs):
        terminal = 0 if int(r["flags"]) & 2 else 1
        internal = int(r["n_stop"]) - terminal
        unamb = int(r["n_codons"]) - int(r["n_ambig"])
        gc = "%.4f" % (int(r["gc"]) / (3.0 * unamb)) if unamb else "."
        gc3 = "%.4f" % (int(r["gc3"]) / float(unamb)) if unamb else "."
        lines.append("\t".join((name, str(int(r["nuc_len"])), str(int(r["n_codons"])), str(int(r["skip"])), str(int(r["rem"])),
                                _codon_text(r["start_codon"]), _codon_text(r["stop_codon"]), str(internal),
                                str(int(r["first_stop"])) if internal > 0 else ".", str(int(r["n_ambig"])), gc, gc3,
                                str(int(r["n_junction"])), str(int(r["n_noncanonical"])), _check_status(r["flags"]))))
    return lines


def _codon_usage_lines(counts, genetic_code):
    """check_cds out_format=codon_usage: the header, then the 64 codons in NCBI order (TTT, TTC, TTA, TTG, TCT, ...): codon,
    residue under the code ('*' = stop), count, per thousand codons counted (2 decimals) and fraction of the codons of the same
    residue (4 decimals); '.' where the denominator is 0.  counts: 64 totals indexed 16*b0 + 4*b1 + b2 (A=0 C=1 G=2 T=3)."""
    counts = [int(c) for c in counts]
    table = gencode.TABLES[gencode.check(genetic_code)]
    total = sum(counts)
    family = {}
    for i, aa in enumerate(table):
        c = "TCAG"[i >> 4] + "TCAG"[(i >> 2) & 3] + "TCAG"[i & 3]
        family[aa] = family.get(aa, 0) + counts["ACGT".index(c[0]) * 16 + "ACGT".index(c[1]) * 4 + "ACGT".index(c[2])]
    lines = [CODON_USAGE_HEADER]
    for i, aa in enumerate(table):
        c = "TCAG"[i >> 4] + "TCAG"[(i >> 2) & 3] + "TCAG"[i & 3]
        n = counts["ACGT".index(c[0]) * 16 + "ACGT".index(c[1]) * 4 + "ACGT".index(c[2])]
        lines.append("\t".join((c, aa, str(n), "%.2f" % (1000.0 * n / total) if total else ".",
                                "%.4f" % (float(n) / family[aa]) if family[aa] else ".")))
    return lines


def check_cds(genome_sequence, gff, feature="gene", genetic_code="1", start_codons="ATG", use_phase="False", out_format="tsv",
              only_ok="False"):
    """Gene-model check of every record `gff2fasta ... seq_type=protein` would print (new): start and stop codon, in-frame
    stops, reading frame, ambiguous codons, GC, splice-site consensus and codon usage, on the device.  start_codons:
    comma-separated codons a CDS may start with (default ATG); use_phase=True starts at the GFF phase of the first CDS;
    genetic_code: NCBI table id.  out_format=tsv prints a header line and one tab-separated line per record (see
    _check_tsv_lines): ID, nuc_len, codons, skip, rem, start, stop, internal_stops, first_internal_stop, ambiguous, gc, gc3,
    junctions, noncanonical, status ('ok' or the comma-joined flags NO_START, NO_STOP, INTERNAL_STOP, PARTIAL_CODON,
    NONCANONICAL_SPLICE, AMBIGUOUS, EMPTY).  out_format=codon_usage prints a header line and the 64 codons in NCBI order (see
    _codon_usage_lines), summed over the records.  only_ok=True keeps only the records without a flag, in both formats."""
    code = gencode.check(genetic_code)
    if out_format not in CHECK_FORMATS:
        raise ValueError("out_format %r is not one of %s" % (out_format, ", ".join(CHECK_FORMATS)))
    codons = start_codons.split(",") if isinstance(start_codons, str) else list(start_codons)
    gencode.start64(codons, code)                            # ValueError before any device work
    phase, ok_only = _truth(use_phase), _truth(only_ok)
    my_genome = genome.Genome(genome_sequence)
    my_genome.read_gff(gff)
    res = my_genome.annotations.check_cds(feature, genetic_code=code, start_codons=codons, use_phase=phase,
                                          codon_usage=out_format == "codon_usage", junctions=False)
    keep = np.flatnonzero(res.records["flags"] == 0) if ok_only else np.arange(len(res.names))
    if out_format == "tsv":
        lines = _check_tsv_lines([res.names[i] for i in keep.tolist()], res.records[keep])
    else:
        lines = _codon_usage_lines(res.codon_counts[keep].sum(axis=0, dtype=np.int64), code)
    sys.stdout.write("\n".join(lines) + "\n")


PREDICT_FORMATS = ("gff3", "protein", "cds")
#: partial= -> (partial5, partial3) of AnnotationSet.predict_cds
PREDICT_PARTIAL = {"none": (False, False), "5prime": (True, False), "3prime": (False, True), "both": (True, True)}
PREDICT_STRANDS = ("sense", "both")


def _predict_header(name, rec, antisense):
    """FASTA header (without '>') of a predicted ORF: <tid>.p1 orf_type=<type> len=<n> <tid>:<lo+1>-<hi>(<+|->), where lo / hi
    are the ORF's coordinates in the transcript ('-': in its reverse complement)."""
    return "%s.p1 orf_type=%s len=%d %s:%d-%d(%s)" % (name, engine._lib.ORF_TYPES[int(rec["type"]) & 3], int(rec["n_aa"]), name,
                                                      int(rec["lo"]) + 1, int(rec["hi"]), "-" if antisense else "+")


def _predict_lines(pred, contig_names, out_format, seqs=None):
    """Output lines of predict_cds for a genome.CdsPrediction.  contig_names[c] = seqid of contig index c; seqs[i] = the protein
    or CDS text of the i-th record that has an ORF (not read for gff3).  gff3: the version line, then per record with an ORF (in
    record order) its CDS segments in ascending start order; protein / cds: a header line and the text on one line."""
    lines = ["##gff-version 3"] if out_format == "gff3" else []
    k = 0
    for i, name in enumerate(pred.names):
        rec = pred.records[i]
        if int(rec["n_aa"]) <= 0:
            continue
        if out_format == "gff3":
            attrs = "ID=%s.cds;Parent=%s;orf_type=%s;length_aa=%d" % (name, name, engine._lib.ORF_TYPES[int(rec["type"]) & 3],
                                                                       int(rec["n_aa"]))
            s0, s1 = int(pred.seg_off[i]), int(pred.seg_off[i + 1])
            for e in sorted(range(s0, s1), key=lambda e: (int(pred.seg_lo[e]), int(pred.seg_hi[e]))):
                lines.append("\t".join((contig_names[int(pred.seg_contig[e])], "magot_b200", "CDS", str(int(pred.seg_lo[e]) + 1),
                                        str(int(pred.seg_hi[e])), ".", "-" if pred.seg_strand[e] else "+",
                                        str(int(pred.seg_phase[e])), attrs)))
        else:
            lines.append(">" + _predict_header(name, rec, pred.antisense[i]))
            lines.append(seqs[k])
        k += 1
    return lines


def _predict_texts(eng, pred, genetic_code, protein):
    """The CDS text (K2) or its translation (K3, trimX off, the first residue 'M' when the ORF starts at a start codon, a
    terminal '*' kept) of every record of `pred` that has an ORF, from one RecordTable of its CDS segments."""
    has = np.flatnonzero(pred.records["n_aa"] > 0)
    if has.size == 0:
        return []
    R = len(pred.names)
    zero = np.zeros(R, dtype=np.int32)
    tbl = engine.RecordTable(pred.seg_off, pred.seg_contig, pred.seg_lo + 1, pred.seg_hi, pred.seg_strand,
                             np.zeros(R, dtype=np.int64), zero, zero, np.zeros(0, dtype=np.uint8))
    text, (nuc_len, aa_len) = eng.run_table(tbl, protein=protein, trimx=False, want_lengths=True,
                                            codon64=gencode.codon64(genetic_code) if protein and genetic_code != 1 else None)
    lens = np.maximum(aa_len, 0) if protein else nuc_len
    off = np.concatenate(([0], np.cumsum(lens)))
    out = []
    for i in has.tolist():
        t = text[off[i]:off[i + 1]].decode("latin-1")
        if protein and not int(pred.records["type"][i]) & 1:
            t = "M" + t[1:]
        out.append(t)
    return out


def predict_cds(genome_sequence, gff, min_orf="100", genetic_code="1", start_codons="ATG", partial="none", strand="sense",
                out_format="gff3"):
    """CDS prediction for exon-only transcript models (new; TransDecoder.LongOrfs / gffread style, one ORF per transcript): the
    longest ORF of each spliced transcript in its three frames, at least `min_orf` residues, from a codon in start_codons
    (comma-separated, default ATG) to a stop of NCBI table `genetic_code`, mapped back to genome CDS segments on the device.
    The GFF is read with exons as the transcripts' base features and CDS rows ignored.  partial=5prime / 3prime / both also
    accept ORFs open at a frame's 5' end / without a stop; strand=both also scores the antisense (the longer ORF wins, the
    sense one on a tie).  out_format: gff3 (CDS rows ID=<tid>.cds;Parent=<tid>;orf_type=..;length_aa=.., segments in
    ascending start order), protein ('>'<tid>.p1 header, the first residue M at a start codon, a terminal '*' kept) or cds
    (the CDS nucleotides under the same header)."""
    code = gencode.check(genetic_code)
    if out_format not in PREDICT_FORMATS:
        raise ValueError("out_format %r is not one of %s" % (out_format, ", ".join(PREDICT_FORMATS)))
    if partial not in PREDICT_PARTIAL:
        raise ValueError("partial %r is not one of %s" % (partial, ", ".join(PREDICT_PARTIAL)))
    if strand not in PREDICT_STRANDS:
        raise ValueError("strand %r is not one of %s" % (strand, ", ".join(PREDICT_STRANDS)))
    try:
        min_aa = int(min_orf)
    except (TypeError, ValueError):
        min_aa = -1
    if min_aa < 0:
        raise ValueError("min_orf %r is not a count of residues" % (min_orf,))
    codons = start_codons.split(",") if isinstance(start_codons, str) else list(start_codons)
    gencode.start64(codons, code)                            # ValueError before any device work
    my_genome = genome.Genome(genome_sequence)
    my_genome.read_gff(gff, base_features=["exon"], features_to_ignore=["CDS"])
    p5, p3 = PREDICT_PARTIAL[partial]
    pred = my_genome.annotations.predict_cds("gene", min_aa=min_aa, genetic_code=code, start_codons=codons, partial5=p5,
                                             partial3=p3, strand=strand)
    gs = my_genome.genome_sequence
    names = {gs.contig_index(seq): seq for seq in gs}
    seqs = None if out_format == "gff3" else _predict_texts(gs._engine(), pred, code, out_format == "protein")
    lines = _predict_lines(pred, names, out_format, seqs)
    sys.stdout.write("\n".join(lines) + "\n" if lines else "")


VARIANT_FORMATS = ("tsv", "vcf")
VARIANT_TSV_HEADER = "\t".join(("CHROM", "POS", "ID", "REF", "ALT", "record", "strand", "consequence", "nuc_pos", "codon",
                                "codons", "residues"))
VARIANT_INFO_HEADER = ('##INFO=<ID=MGCSQ,Number=.,Type=String,Description="Coding consequence per allele and record: '
                       'class|allele|record|strand|ref_aa/alt_aa|1-based payload position">')


def _codon_text(c):
    return "." if c == 0xFF else "ACGT"[c >> 4] + "ACGT"[(c >> 2) & 3] + "ACGT"[c & 3]


def _variant_fields(res, k):
    """(consequence, strand, 1-based payload position, 1-based codon, codons, residues) of row k of a genome.VariantEffects;
    '.' for an absent value."""
    row = res.rows[k]
    cls = engine._lib.VEF_CLASSES[int(row["cls"]) - 1]
    nuc = "." if int(row["nuc_lo"]) < 0 else str(int(row["nuc_lo"]) + 1)
    codon = "." if int(row["codon"]) < 0 else str(int(row["codon"]) + 1)
    n_aff = int(row["n_aff"])
    codons = "." if n_aff == 0 else "%s/%s" % (_codon_text(int(row["ref_codon"])), _codon_text(int(row["alt_codon"])))
    aa = "." if n_aff == 0 else "%s/%s" % (bytes(row["ref_aa"]).decode("latin-1"), bytes(row["alt_aa"]).decode("latin-1"))
    return cls, "-" if res.strand[k] else "+", nuc, codon, codons, aa


def variant_effects(genome_sequence, gff, vcf, feature="gene", genetic_code="1", start_codons="ATG", use_phase="False",
                    out_format="tsv"):
    """Coding consequences of the alleles of a VCF (plain or gzip) on every record `check_cds` checks (new; bcftools csq /
    SnpEff style, on the device): splice acceptor or donor site, segment boundary, frameshift, in-frame insertion or deletion,
    start lost, stop gained, stop lost, ambiguous, missense, synonymous, or a substitution outside the codons.  Multi-allelic
    lines give one allele per ALT; symbolic, '*', '.' and breakend ALTs are skipped.  out_format=tsv prints a header line and
    one line per (allele, record): CHROM, POS, ID, REF, ALT, record, strand of the owning segment, consequence, 1-based
    payload position, 1-based codon, codons (GCT/GTT) and residues (A/V) of a substitution's first affected codon(s), '.' when
    absent.  out_format=vcf prints the VCF unchanged except for an ##INFO=<ID=MGCSQ> header line and, on lines with rows,
    MGCSQ=class|allele|record|strand|aa_change|nuc_pos entries added to INFO.  The status counts (0 ok, 1 unknown contig or
    out of range, 2 REF mismatch, 3 empty or REF == ALT) and the skipped ALTs go to stderr."""
    code = gencode.check(genetic_code)
    if out_format not in VARIANT_FORMATS:
        raise ValueError("out_format %r is not one of %s" % (out_format, ", ".join(VARIANT_FORMATS)))
    codons = start_codons.split(",") if isinstance(start_codons, str) else list(start_codons)
    gencode.start64(codons, code)                            # ValueError before any device work
    phase = _truth(use_phase)
    from . import variants as _variants
    calls = _variants.read_vcf(vcf)
    my_genome = genome.Genome(genome_sequence)
    my_genome.read_gff(gff)
    res = my_genome.annotations.variant_effects(feature, calls, genetic_code=code, start_codons=codons, use_phase=phase)
    out = []
    if out_format == "tsv":
        out.append(VARIANT_TSV_HEADER)
        for k in range(res.rows.size):
            i = int(res.rows["var"][k])
            f = _variant_fields(res, k)
            out.append("\t".join((calls.chrom[i], str(int(calls.pos[i])), calls.ids[i], calls.ref[i].decode("latin-1"),
                                  calls.alt[i].decode("latin-1"), res.names[int(res.rows["rec"][k])], f[1], f[0], f[2], f[3],
                                  f[4], f[5])))
    else:
        per_line = {}
        for k in range(res.rows.size):
            i = int(res.rows["var"][k])
            cls, strand, nuc, _, _, aa = _variant_fields(res, k)
            per_line.setdefault(int(calls.line[i]), []).append(
                "|".join((cls, calls.alt[i].decode("latin-1"), res.names[int(res.rows["rec"][k])], strand,
                          "" if aa == "." else aa, "" if nuc == "." else nuc)))
        header_done = False
        for n, text in enumerate(calls.lines):
            line = text.decode("latin-1")
            if line.startswith("#CHROM") and not header_done:
                out.append(VARIANT_INFO_HEADER)
                header_done = True
            if n in per_line:
                cols = line.split("\t")
                while len(cols) < 8:
                    cols.append(".")
                entry = "MGCSQ=" + ",".join(per_line[n])
                cols[7] = entry if cols[7] in ("", ".") else cols[7] + ";" + entry
                line = "\t".join(cols)
            out.append(line)
    sys.stdout.write("\n".join(out) + "\n")
    counts = np.bincount(res.status.astype(np.int64), minlength=4) if res.status.size else np.zeros(4, np.int64)
    sys.stderr.write("variant_effects: %d alleles, status ok %d, unknown contig or out of range %d, REF mismatch %d, "
                     "empty or unchanged %d; skipped ALTs: %s; %d rows\n"
                     % (len(calls), counts[0], counts[1], counts[2], counts[3],
                        ", ".join("%s %d" % kv for kv in calls.skipped.items()), res.rows.size))


FUNCTIONS = {f.__name__: f for f in (gff2fasta, cds2pep, coords2fasta, get_seq_from_fasta, exclude_from_fasta,
                                     extract_upstream_downstream, dna2orfs, blast_csv2fasta, exonerate2fasta, mask_from_gff,
                                     convert_gff, call_orfs, check_cds, predict_cds, variant_effects)}


def help_func():
    print("\ngenome_tools script from MAGOT (B200 path).\n\nUsage: " + sys.argv[0] +
          " function [option1=<option1 choice> ...] \n\nFunctions:\n    " + '\n    '.join(sorted(FUNCTIONS)))


def main(argv=None):
    """genome_tools.py:25-45 -- same grammar: `name=value` -> keyword argument (value = text between the
    first and second '='), anything else positional; all values are strings."""
    argv = sys.argv if argv is None else argv
    program = argv[1]
    arguments = argv[2:]
    if program in ('-h', '-help', '--help', 'help'):
        help_func()
        return None
    if len(arguments) > 0 and arguments[0] in ('-h', '--help', '-help', 'help', '--h'):
        print('hey')
        return None
    if program not in FUNCTIONS:
        raise NameError("name %r is not defined" % program)
    args, kwargs = [], {}
    for argument in arguments:
        if '=' in argument:
            argsplit = argument.split('=')
            kwargs[argsplit[0]] = argsplit[1]
        else:
            args.append(argument)
    return FUNCTIONS[program](*args, **kwargs)


if __name__ == "__main__":
    main()
