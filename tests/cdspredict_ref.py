"""Test helper: an independent statement of the CDS prediction (mg_plan_predict_cds*, engine.Plan.predict_cds,
AnnotationSet.predict_cds, genome_tools predict_cds) in numpy / pure Python.

It does not import magot_b200.  Record r's payload S is cdscheck_ref.payload (clamped segments in emission order, each
reverse-complemented by its strand).  A codon starts at every i with i + 3 <= len(S); its frame is i mod 3.  In each frame the
stops cut the codons into stretches; a stretch's ORF runs from its first start codon (with partial5, the first stretch of a
frame from its first codon) through the stop, or, with partial3, through the frame's last complete codon when the stretch has
no stop.  A candidate needs n_aa >= max(1, min_aa); the record's ORF is the candidate with the most residues, then the
smallest start.  Codon indices are 16*b0 + 4*b1 + b2 with A=0 C=1 G=2 T=3; 0xFF is an absent or ambiguous codon.
"""
import numpy as np

import cdscheck_ref as cref
import gencode_ref as gref

FIELDS = ("lo", "hi", "n_aa", "frame", "type", "start_codon", "stop_codon", "n_cds_seg")
ORF_TYPES = ("complete", "5prime_partial", "3prime_partial", "internal")
NONE = dict(lo=-1, hi=-1, n_aa=0, frame=-1, type=0, start_codon=0xFF, stop_codon=0xFF, n_cds_seg=0)

_BASE = np.full(256, -1, dtype=np.int64)
for _i, _c in enumerate(b"ACGT"):
    _BASE[_c] = _i
    _BASE[ord(chr(_c).lower())] = _i


def codon_indices(S):
    """Index of the codon at every position i with i + 3 <= len(S), -1 where a base is outside A/C/G/T."""
    b = _BASE[np.frombuffer(bytes(S), dtype=np.uint8)]
    if b.size < 3:
        return np.zeros(0, dtype=np.int64)
    idx = b[:-2] * 16 + b[1:-1] * 4 + b[2:]
    idx[(b[:-2] < 0) | (b[1:-1] < 0) | (b[2:] < 0)] = -1
    return idx


def code_sets(code, starts):
    """(stop flags, start flags) as boolean arrays of 64 under NCBI table `code` and the start codons `starts`."""
    table = gref.table64(code)
    stop = np.array([a == "*" for a in table])
    start = np.zeros(64, dtype=bool)
    for c in starts:
        start[cref.codon_index(c.upper().encode())] = True
    return stop, start


def candidates(S, stop, start, partial5=False, partial3=False):
    """Every stretch's ORF of payload S, before the min_aa filter: list of (n_aa, lo, hi, has_stop)."""
    idx = codon_indices(S)
    out = []
    for f in range(3):
        pos = np.arange(f, idx.size, 3)
        if pos.size == 0:
            continue
        c = idx[pos]
        ok = c >= 0
        is_stop = ok & stop[np.maximum(c, 0)]
        is_start = ok & start[np.maximum(c, 0)] & ~is_stop
        sp, st = pos[is_stop], pos[is_start]
        begins = np.concatenate(([f], sp + 3))
        ends = np.concatenate((sp, [np.iinfo(np.int64).max]))        # the last stretch is open at its 3' end
        j = np.searchsorted(st, begins)
        first = np.where(j < st.size, st[np.minimum(j, max(st.size - 1, 0))] if st.size else 0, -1)
        first = np.where((first >= 0) & (first < ends), first, -1)
        if partial5:
            first[0] = f
        for k in range(sp.size):
            if first[k] >= 0:
                out.append(((int(sp[k]) - int(first[k])) // 3, int(first[k]), int(sp[k]) + 3, True))
        if partial3 and first[-1] >= 0:
            hi = int(pos[-1]) + 3
            out.append(((hi - int(first[-1])) // 3, int(first[-1]), hi, False))
    return out


def select(cands, min_aa):
    """The chosen candidate (n_aa, lo, hi, has_stop) or None."""
    keep = [c for c in cands if c[0] >= max(1, min_aa)]
    if not keep:
        return None
    return max(keep, key=lambda c: (c[0], -c[1]))


def orf_record(S, orf, start):
    """The mg_cds_pred fields (n_cds_seg left 0) of an ORF of payload S."""
    if orf is None:
        return dict(NONE)
    n_aa, lo, hi, has_stop = orf
    sc = cref.codon_index(S[lo:lo + 3])
    sc = 0xFF if sc is None else sc
    ec = 0xFF
    if has_stop:
        ec = cref.codon_index(S[hi - 3:hi])
    t = (0 if sc != 0xFF and start[sc] else 1) | (0 if has_stop else 2)
    return dict(lo=lo, hi=hi, n_aa=n_aa, frame=lo % 3, type=t, start_codon=sc, stop_codon=ec, n_cds_seg=0)


def clamped_segments(contigs, tbl, r):
    """[(cl, ch, minus)] of the segments of record r, clamped as the plan clamps them (empty for a contig outside the genome)."""
    out = []
    for e in range(int(tbl.rec_seg_off[r]), int(tbl.rec_seg_off[r + 1])):
        c = int(tbl.seg_contig[e])
        if c < 0 or c >= len(contigs):
            out.append((0, 0, bool(tbl.seg_strand[e])))
            continue
        a, b = cref.clamp(len(contigs[c]), tbl.seg_start[e], tbl.seg_end[e])
        out.append((a, b, bool(tbl.seg_strand[e])))
    return out


def map_segments(segs, lo, hi):
    """[(lo, hi, phase)] per segment: the forward-contig interval of the segment's share of payload range [lo, hi), (-1, -1, -1)
    where the range does not touch it."""
    out = []
    o = 0
    for cl, ch, minus in segs:
        ln = ch - cl
        x, y = max(lo, o), min(hi, o + ln)
        if lo >= 0 and x < y:
            a, b = (ch - (y - o), ch - (x - o)) if minus else (cl + x - o, cl + y - o)
            out.append((a, b, (3 - (x - lo) % 3) % 3))
        else:
            out.append((-1, -1, -1))
        o += ln
    return out


def predict(contigs, tbl, code=1, starts=("ATG",), min_aa=0, partial5=False, partial3=False, cache=None):
    """(records: list of dicts with FIELDS, segments: list of (lo, hi, phase) per segment of tbl).  `cache` (a dict) keeps the
    payloads and the candidates across calls that differ in min_aa only."""
    stop, start = code_sets(code, starts)
    cache = {} if cache is None else cache
    key = (code, tuple(starts), bool(partial5), bool(partial3))
    if "payload" not in cache:
        cache["payload"] = [cref.payload(contigs, tbl, r) for r in range(tbl.n_rec)]
    if key not in cache:
        cache[key] = [candidates(S, stop, start, partial5, partial3) for S in cache["payload"]]
    recs, segs = [], []
    for r in range(tbl.n_rec):
        S = cache["payload"][r]
        rec = orf_record(S, select(cache[key][r], min_aa), start)
        m = map_segments(clamped_segments(contigs, tbl, r), rec["lo"], rec["hi"])
        rec["n_cds_seg"] = sum(1 for s in m if s[0] >= 0)
        recs.append(rec)
        segs.extend(m)
    return recs, segs


def antisense(tbl):
    """Columns (rec_seg_off, seg_contig, seg_start, seg_end, seg_strand) of the antisense table of tbl: each record's segments
    in reverse order with their strands flipped, so that its payload is the reverse complement of the record's."""
    order = []
    for r in range(tbl.n_rec):
        order.extend(range(int(tbl.rec_seg_off[r + 1]) - 1, int(tbl.rec_seg_off[r]) - 1, -1))
    order = np.array(order, dtype=np.int64)
    return (np.asarray(tbl.rec_seg_off), np.asarray(tbl.seg_contig)[order], np.asarray(tbl.seg_start)[order],
            np.asarray(tbl.seg_end)[order], (np.asarray(tbl.seg_strand)[order] == 0).astype(np.int8))


def compare(got_recs, got_segs, want_recs, want_segs):
    """Field-by-field comparison of PRED_DTYPE / CDSSEG_DTYPE arrays (got_segs may be None) with predict(); first mismatch or None."""
    if len(got_recs) != len(want_recs):
        return "%d records, want %d" % (len(got_recs), len(want_recs))
    for r, w in enumerate(want_recs):
        for f in FIELDS:
            if int(got_recs[f][r]) != w[f]:
                return "record %d field %s: %d, want %d (want %s)" % (r, f, int(got_recs[f][r]), w[f], w)
    if got_segs is not None:
        if len(got_segs) != len(want_segs):
            return "%d segments, want %d" % (len(got_segs), len(want_segs))
        for e, w in enumerate(want_segs):
            g = (int(got_segs["lo"][e]), int(got_segs["hi"][e]), int(got_segs["phase"][e]))
            if g != tuple(w):
                return "segment %d: %s, want %s" % (e, g, tuple(w))
    return None
