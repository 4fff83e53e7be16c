"""Test helper: an independent statement of the variant consequence call (mg_plan_variant_count / _emit, engine.Plan.
variant_effects, AnnotationSet.variant_effects) in pure Python.

It works from host genome bytes (one bytes object per contig), a RecordTable and a list of alleles (contig, pos, ref, alt)
sorted by (contig, pos); it does not import magot_b200.  The rules are the ones include/magot_b200.h states: status, the
suffix-then-prefix trim, touch, the owning segment, the class and the codon fields.  Row fields are those of VEF_DTYPE, with
ref_aa / alt_aa as bytes without the NUL padding.
"""
import bisect

import numpy as np

import cdscheck_ref as cref
import gencode_ref as gref

(SPLICE_ACCEPTOR, SPLICE_DONOR, BOUNDARY, FRAMESHIFT, INFRAME_INSERTION, INFRAME_DELETION, START_LOST, STOP_GAINED, STOP_LOST,
 AMBIGUOUS, MISSENSE, SYNONYMOUS, NONCODING_PAYLOAD) = range(1, 14)
FIELDS = ("var", "rec", "seg", "nuc_lo", "nuc_hi", "codon", "cls", "n_aff", "ref_codon", "alt_codon", "ref_aa", "alt_aa")
_PACKED = set(b"ACGTacgtNn-RYKM")           # genome bytes held in the packed planes; any other byte is an exception
_COMP = {ord("A"): ord("T"), ord("C"): ord("G"), ord("G"): ord("C"), ord("T"): ord("A")}


def _up(b):
    return bytes(b).upper()


def normalise(pos, ref, alt):
    """(s, t, A'): forward span of REF' and the remaining ALT bytes after the suffix-then-prefix trim (case ignored)."""
    R, A = _up(ref), _up(alt)
    m = min(len(R), len(A))
    suf = 0
    while suf < m and R[len(R) - 1 - suf] == A[len(A) - 1 - suf]:
        suf += 1
    pre = 0
    while pre < m - suf and R[pre] == A[pre]:
        pre += 1
    return pos + pre, pos + len(R) - suf, bytes(alt)[pre:len(alt) - suf]


def status(contigs, c, pos, ref, alt):
    if c < 0 or c >= len(contigs) or pos < 0 or pos + len(ref) > len(contigs[c]):
        return 1
    g = contigs[c][pos:pos + len(ref)]
    for gb, rb in zip(g, bytes(ref)):
        if gb not in _PACKED or _up(bytes([gb])) != _up(bytes([rb])):
            return 2
    if not ref or not alt or _up(ref) == _up(alt):
        return 3
    return 0


def segments(contigs, tbl, r):
    """[(e, contig, cl, ch, minus)] of record r, clamped as the plan clamps them (an unknown contig gives an empty segment)."""
    out = []
    for e in range(int(tbl.rec_seg_off[r]), int(tbl.rec_seg_off[r + 1])):
        c = int(tbl.seg_contig[e])
        cl = ch = 0
        if 0 <= c < len(contigs):
            cl, ch = cref.clamp(len(contigs[c]), tbl.seg_start[e], tbl.seg_end[e])
        out.append((e, c, cl, ch, bool(tbl.seg_strand[e])))
    return out


def sites(x, y):
    """((donor u, shared point), (acceptor u, shared point)) of the junction between segments x and y, or None (class 0)."""
    _, c0, a0, b0, m0 = x
    _, c1, a1, b1, m1 = y
    if b0 <= a0 or b1 <= a1 or c0 != c1 or m0 != m1:
        return None
    if not m0:
        return ((b0, b0), (a1 - 2, a1)) if a1 - b0 >= 4 else None
    return ((a0 - 2, a0), (b1, b1)) if a0 - b1 >= 4 else None


def _payload_base(contigs, segs, offs):
    """base(q): byte q of the record's payload (its clamped segments in order, '-' ones reverse-complemented as
    gencode_ref.revcomp does), read without building the payload."""
    def base(q):
        k = int(np.searchsorted(offs, q, side="right")) - 1      # the last segment starting at or before q: not empty
        _, c, cl, ch, minus = segs[k]
        if minus:
            return gref.revcomp(contigs[c][ch - 1 - (q - offs[k]):ch - (q - offs[k])])[0]
        return contigs[c][cl + q - offs[k]]
    return base


def touch_interval(s, t, u, w):
    return s < w and u < t


def touch_site(s, t, site):
    u, sh = site
    return touch_interval(s, t, u, u + 2) if t > s else (s == u + 1 or s == sh)


def touch_seg(s, t, seg):
    _, _, cl, ch, _ = seg
    return touch_interval(s, t, cl, ch) if t > s else cl < s < ch


def effects(contigs, tbl, alleles, code=1, starts=("ATG",), use_phase=False):
    """(status list, row dicts ordered by record, then allele) for alleles [(contig, pos, ref, alt)] sorted by (contig, pos)."""
    table = gref.table64(code)
    stop = [a == "*" for a in table]
    start = set(cref.codon_index(x.upper().encode()) for x in starts)
    st = [status(contigs, c, p, ref, alt) for c, p, ref, alt in alleles]
    norm = [normalise(p, ref, alt) if s == 0 else None for (c, p, ref, alt), s in zip(alleles, st)]
    keys = [(c, p) for c, p, _, _ in alleles]
    max_ref = max([len(a[2]) for a, s in zip(alleles, st) if s == 0] + [0])
    rows = []
    for r in range(tbl.n_rec):
        segs = segments(contigs, tbl, r)
        cand = set()                                   # alleles that can touch the record: pos in [cl - 3 - max_ref, ch + 3)
        for _, c, cl, ch, _ in segs:
            cand.update(range(bisect.bisect_left(keys, (c, cl - 3 - max_ref)), bisect.bisect_left(keys, (c, ch + 3))))
        junc = [sites(segs[k], segs[k + 1]) if k + 1 < len(segs) else None for k in range(len(segs))]
        offs = np.concatenate(([0], np.cumsum([ch - cl for _, _, cl, ch, _ in segs]))).astype(np.int64)
        base = _payload_base(contigs, segs, offs)
        skip = 0
        if use_phase and tbl.rec_phase is not None and 0 <= int(tbl.rec_phase[r]) <= 2:
            skip = int(tbl.rec_phase[r])
        L = int(offs[-1]) - skip
        ncod = L // 3 if L > 0 else 0
        for i in sorted(cand):
            c, p, ref, alt = alleles[i]
            if st[i]:
                continue
            s, t, A = norm[i]
            owner = None
            acc = don = inside = False
            for k, seg in enumerate(segs):
                if seg[1] != c:
                    continue
                hit = touch_seg(s, t, seg)
                if junc[k] is not None:
                    d, a = touch_site(s, t, junc[k][0]), touch_site(s, t, junc[k][1])
                    don, acc, hit = don or d, acc or a, hit or d or a
                if hit and owner is None:
                    owner = k
                if (t > s and seg[2] <= s and t <= seg[3]) or (t == s and seg[2] < s < seg[3]):
                    inside = True
            if owner is None:
                continue
            e, _, cl, ch, minus = segs[owner]
            o = int(offs[owner])
            nlo = nhi = -1
            if t > s:
                x0, x1 = max(s, cl), min(t, ch)
                if x0 < x1:
                    nlo, nhi = (o + ch - x1, o + ch - x0) if minus else (o + x0 - cl, o + x1 - cl)
            elif cl < s < ch:
                nlo = nhi = o + ch - s if minus else o + s - cl
            sub = t - s == len(A)
            row = dict(var=i, rec=r, seg=e, nuc_lo=nlo, nuc_hi=nhi, codon=-1, cls=0, n_aff=0, ref_codon=0xFF, alt_codon=0xFF,
                       ref_aa=b"", alt_aa=b"")
            aff = []
            if nlo >= 0:
                if sub:
                    x0, x1 = max(nlo, skip), min(nhi, skip + 3 * ncod)      # codons k < ncod overlapping [nlo, nhi)
                    aff = list(range((x0 - skip) // 3, (x1 - 1 - skip) // 3 + 1)) if x0 < x1 else []
                    if aff:
                        row["codon"] = aff[0]
                elif skip <= nlo < skip + 3 * ncod:
                    row["codon"] = (nlo - skip) // 3
            if acc:
                cls = SPLICE_ACCEPTOR
            elif don:
                cls = SPLICE_DONOR
            elif not inside:
                cls = BOUNDARY
            elif not sub:
                d = len(A) - (t - s)
                cls = FRAMESHIFT if d % 3 else (INFRAME_INSERTION if d > 0 else INFRAME_DELETION)
            elif not aff:
                cls = NONCODING_PAYLOAD
            else:
                put = bytes(A)
                if minus:
                    put = bytes(_COMP.get(b, ord("N")) for b in _up(put)[::-1])

                def codons(k):                     # (reference, alternative) codon index of codon k
                    q = range(skip + 3 * k, skip + 3 * k + 3)
                    ref_c = bytes(base(x) for x in q)
                    alt_c = bytes(put[x - nlo] if nlo <= x < nhi else base(x) for x in q)
                    return cref.codon_index(ref_c), cref.codon_index(alt_c)

                flags = set()
                ra, aa = [], []
                for k in aff:
                    rc, ac = codons(k)
                    rres = "X" if rc is None else table[rc]
                    ares = "X" if ac is None else table[ac]
                    if k == 0 and rc is not None and rc in start and not (ac is not None and ac in start):
                        flags.add(START_LOST)
                    if rc is not None and not stop[rc] and ac is not None and stop[ac]:
                        flags.add(STOP_GAINED)
                    if k == ncod - 1 and rc is not None and stop[rc] and not (ac is not None and stop[ac]):
                        flags.add(STOP_LOST)
                    if rc is None or ac is None:
                        flags.add(AMBIGUOUS)
                    elif rres != ares:
                        flags.add(MISSENSE)
                    ra.append(rres)
                    aa.append(ares)
                cls = min(flags) if flags else SYNONYMOUS
                rc0, ac0 = codons(aff[0])
                row.update(n_aff=min(len(aff), 127), ref_codon=0xFF if rc0 is None else rc0, alt_codon=0xFF if ac0 is None else ac0,
                           ref_aa="".join(ra[:8]).encode(), alt_aa="".join(aa[:8]).encode())
            row["cls"] = cls
            rows.append(row)
    return st, rows


def compare(status_got, rows_got, status_want, rows_want):
    """Field-by-field comparison of device results (int8 status, VEF_DTYPE rows) with effects(); first mismatch or None."""
    if list(np.asarray(status_got).tolist()) != list(status_want):
        bad = [i for i, (a, b) in enumerate(zip(np.asarray(status_got).tolist(), status_want)) if a != b][:5]
        return "status differs at alleles %s (of %d / %d)" % (bad, len(status_got), len(status_want))
    if len(rows_got) != len(rows_want):
        return "%d rows, want %d" % (len(rows_got), len(rows_want))
    for k, w in enumerate(rows_want):
        for f in FIELDS:
            g = rows_got[f][k]
            g = bytes(g) if f in ("ref_aa", "alt_aa") else int(g)
            if g != w[f]:
                return "row %d (allele %d, record %d) field %s: %r, want %r" % (k, w["var"], w["rec"], f, g, w[f])
    return None
