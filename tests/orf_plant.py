"""Test helper: sequences with ORFs planted at exact positions, and what each plant is meant to give.

It does not import magot_b200.  The background is drawn from an alphabet that holds no stop and no start codon in any frame
under the codes the suites use (1, 2, 6, 11, 23) and the start sets ATG and {ATG, GTG, TTG}: A/C for a payload read on one
strand, C/G for a contig read on both (its reverse complement is C/G again; that of A/C is G/T, full of GTG and TTG).  Under
the "sense" start set every codon outside a stop and an N run is a start, and the intent says so.  Each planted codon gets
the one-base flanks that keep every codon overlapping it, on both strands when asked, free of stops and starts; Strand.verify
scans the finished sequence and fails when it holds a stop or a start codon that was not planted.

The case generators at the end build the planted genomes of tests/test_host_orf_edges.py (which checks each intent against
the references) and tests/test_gpu_orf_edges.py (which runs them on the device).  Positions are 0-based offsets of a codon's
first base on the strand it is read on.  intent() restates, from the planted
codons alone, the stretch rule of the headers (include/magot_b200.h): per frame the stops cut the codons into stretches, a
stretch's ORF runs from its first start through its stop, or, open at the 3' end, through the frame's last complete codon.
"""
import itertools

import numpy as np

import gencode_ref as gref

SENSE = "sense"
_IDX = {b: i for i, b in enumerate(b"ACGT")}
_IDX.update({b + 32: i for b, i in list(_IDX.items())})


def _codon(s):
    """Index 16*b0 + 4*b1 + b2 of 3 bytes, None when one is outside A/C/G/T."""
    try:
        return _IDX[s[0]] * 16 + _IDX[s[1]] * 4 + _IDX[s[2]]
    except KeyError:
        return None


def stops_of(code):
    """The stop codons of NCBI table `code`, upper case."""
    t = gref.table64(code)
    return ["ACGT"[i >> 4] + "ACGT"[(i >> 2) & 3] + "ACGT"[i & 3] for i in range(64) if t[i] == "*"]


def clean_stop(code, alphabet=b"AC", both=False, k=0):
    """The k-th (cyclically) stop codon of `code` that can be planted cleanly on `alphabet` (on both strands when `both`:
    under code 23 TAA reads TTA, a stop, on the other strand)."""
    ok = []
    for c in stops_of(code):
        try:
            _flanks(c, alphabet, code, SENSE, both)
            ok.append(c)
        except ValueError:
            pass
    return ok[k % len(ok)]


def start_set(code, which):
    """The start codons of `which` (a tuple, or SENSE: every codon that is no stop under `code`)."""
    if which != SENSE:
        return tuple(which)
    stop = set(stops_of(code))
    return tuple(c for c in ("ACGT"[i >> 4] + "ACGT"[(i >> 2) & 3] + "ACGT"[i & 3] for i in range(64)) if c not in stop)


def _flags(code, starts):
    stop = np.zeros(64, dtype=bool)
    for c in stops_of(code):
        stop[_codon(c.encode())] = True
    start = np.zeros(64, dtype=bool)
    if starts != SENSE:
        for c in starts:
            start[_codon(c.upper().encode())] = True
    return stop, start & ~stop


_BASE = np.full(256, -1, dtype=np.int64)
for _b, _i in _IDX.items():
    _BASE[_b] = _i


def events(seq, code, starts, minus=False):
    """{(pos, kind)} of the stop ('*') and start ('M') codons of bytes `seq` read on its plus strand (or, minus=True, its
    reverse complement); starts == SENSE lists stops only."""
    s = gref.revcomp(seq) if minus else seq
    stop, start = _flags(code, starts)
    b = _BASE[np.frombuffer(bytes(s), dtype=np.uint8)]
    if b.size < 3:
        return set()
    idx = b[:-2] * 16 + b[1:-1] * 4 + b[2:]
    ok = (b[:-2] >= 0) & (b[1:-1] >= 0) & (b[2:] >= 0)
    idx = np.where(ok, idx, 0)
    return ({(int(i), "*") for i in np.flatnonzero(ok & stop[idx])} |
            {(int(i), "M") for i in np.flatnonzero(ok & start[idx])})


_FLANK_CACHE = {}


def _flanks(codon, alphabet, code, starts, both):
    """(left, right) bases around `codon` such that no codon overlapping it but itself is a stop or a start, whatever
    background bases of `alphabet` surround them, on the read strand (and its reverse complement when `both`)."""
    key = (codon, alphabet, code, starts if starts == SENSE else tuple(starts), both)
    if key in _FLANK_CACHE:
        return _FLANK_CACHE[key]
    want = "*" if codon in stops_of(code) else ("M" if starts != SENSE and codon in starts else None)
    for l, r in itertools.product(b"CAGT", repeat=2):
        ok = True
        for bg in itertools.product(alphabet, repeat=6):
            s = bytes(bg[:3]) + bytes([l]) + codon.encode() + bytes([r]) + bytes(bg[3:])
            ev = events(s, code, starts)
            if ev - {(4, want)} or (want and (4, want) not in ev):
                ok = False
                break
            if both:
                e2 = {(len(s) - 3 - p, k) for p, k in events(s, code, starts, minus=True)}
                if e2:
                    ok = False
                    break
        if ok:
            _FLANK_CACHE[key] = (l, r)
            return l, r
    raise ValueError("no flanks keep %s clean under code %d" % (codon, code))


class Strand:
    """A sequence of n bases read on one strand, with planted codons.  alphabet: the background bases; both: keep the
    reverse complement clean too (a contig, read on both strands).  Plants on the minus strand (both only) are given as read
    there, at minus-strand offsets."""

    def __init__(self, n, rng, code, starts, alphabet=b"AC", both=False):
        self.n, self.code, self.starts, self.both = n, code, starts, both
        self.alphabet = alphabet
        self.buf = bytearray(np.frombuffer(alphabet, dtype=np.uint8)[rng.integers(0, len(alphabet), size=n)].tobytes())
        self.fixed = {}                                # forward position -> base a plant or a flank needs
        self.plants = {0: [], 1: []}                   # minus -> [(pos, codon)]
        self.nruns = []                                # forward [a, b)

    def _put(self, x, b, codon):
        """Base b at forward x: a codon base may overwrite a flank, nothing else may change a fixed base."""
        if not 0 <= x < self.n:
            return
        old = self.fixed.get(x)
        if old is not None and old[0] != b and (not codon or old[1]):
            if not codon:
                return                                   # a flank next to another plant's codon: verify() judges it
            raise ValueError("plant at %d collides with another plant" % x)
        self.fixed[x] = (b, codon)
        self.buf[x] = b

    def plant(self, pos, codon, minus=False):
        """Put `codon` (as read on its strand) at offset `pos` of that strand."""
        assert 0 <= pos and pos + 3 <= self.n and (self.both or not minus)
        l, r = _flanks(codon, self.alphabet, self.code, self.starts, self.both)
        c, x = codon.encode(), pos
        if minus:
            c, x = gref.revcomp(c), self.n - pos - 3
            l, r = gref.revcomp(bytes([r]))[0], gref.revcomp(bytes([l]))[0]
        for k in range(3):
            self._put(x + k, c[k], True)
        self._put(x - 1, l, False)
        self._put(x + 3, r, False)
        self.plants[int(minus)].append((pos, codon))
        return self

    def orf(self, lo, n_aa, start="ATG", stop=None, minus=False):
        """A start codon at lo, n_aa - 1 background codons, then `stop` (None: the code's first stop, False: no stop)."""
        self.plant(lo, start, minus)
        if stop is not False:
            self.plant(lo + 3 * n_aa, stop or stops_of(self.code)[0], minus)
        return self

    def n_run(self, a, b):
        """N over forward [a, b), clear of every planted base."""
        for x in range(a, b):
            assert x not in self.fixed
            self.buf[x] = ord("N")
        self.nruns.append((a, b))
        return self

    def seq(self, rng=None):
        """The bases; with rng, a random half of them in lower case."""
        s = bytes(self.buf)
        if rng is None:
            return s
        low = rng.integers(0, 2, size=self.n).astype(bool)
        a = np.frombuffer(s, dtype=np.uint8).copy()
        a[low & (a != ord("N"))] += 32
        return a.tobytes()

    def verify(self):
        """Fail unless the stops and starts of the sequence are exactly the planted ones (stops only under SENSE)."""
        for m in ((0, 1) if self.both else (0,)):
            want = set()
            for pos, c in self.plants[m]:
                if c in stops_of(self.code):
                    want.add((pos, "*"))
                elif self.starts != SENSE and c in self.starts:
                    want.add((pos, "M"))
            got = events(bytes(self.buf), self.code, self.starts, bool(m))
            assert got == want, ("minus" if m else "plus", sorted(got ^ want)[:6])
        return self

    def _ncodon(self, minus):
        """Offsets on the strand of the codons that hold an N."""
        bad = set()
        for a, b in self.nruns:
            if minus:
                a, b = self.n - b, self.n - a
            bad.update(range(max(0, a - 2), b))
        return bad

    def intent(self, minus=False, partial5=False, partial3=False):
        """Every stretch's ORF on the strand as planned: [(n_aa, lo, hi, has_stop)], lo / hi strand offsets."""
        stop_set = set(stops_of(self.code))
        stops = {p for p, c in self.plants[int(minus)] if c in stop_set}
        if self.starts == SENSE:
            bad = self._ncodon(minus)
            is_start = lambda p: p not in bad and p not in stops          # noqa: E731
        else:
            st = {p for p, c in self.plants[int(minus)] if c in self.starts and c not in stop_set}
            is_start = st.__contains__
        out = []
        for f in range(3):
            m = (self.n - f) // 3 if self.n > f else 0
            first = f if partial5 else None
            for k in range(m):
                p = f + 3 * k
                if first is None and is_start(p):
                    first = p
                if p in stops:
                    if first is not None:
                        out.append(((p - first) // 3, first, p + 3, True))
                    first = None
            if partial3 and first is not None:
                hi = f + 3 * m
                out.append(((hi - first) // 3, first, hi, False))
        return out


def winner(cands, min_aa):
    """The chosen candidate of a record: most residues, then the smallest start; None below max(1, min_aa)."""
    keep = [c for c in cands if c[0] >= max(1, min_aa)]
    return max(keep, key=lambda c: (c[0], -c[1])) if keep else None


def calls(strand, min_aa, partial):
    """The ORF calls of a both-strand Strand as planned: [(minus, phase, lo, hi, len, has_stop)] in forward coordinates."""
    out = []
    for m in (0, 1):
        for n_aa, lo, hi, stop in strand.intent(bool(m), False, partial):
            if n_aa >= min_aa:
                flo, fhi = (strand.n - hi, strand.n - lo) if m else (lo, hi)
                out.append((m, lo % 3, flo, fhi, n_aa, stop))
    return sorted(out)


def split(payload, cuts, minus, rng, contig_id):
    """A contig and the segments [(contig_id, start, end, strand)] (1-based, inclusive) whose spliced payload is `payload`
    cut at the payload offsets `cuts`; minus[k] is the strand of piece k (a bool for all).  Random A/C/G/T introns and flanks
    lie between the pieces; the pieces of a record on '-' lie in descending order, as a gene on '-' would."""
    edges = [0] + sorted(cuts) + [len(payload)]
    pieces = [payload[a:b] for a, b in zip(edges[:-1], edges[1:])]
    strands = [bool(minus)] * len(pieces) if isinstance(minus, (bool, int)) else [bool(x) for x in minus]
    order = list(range(len(pieces)))
    if all(strands):
        order.reverse()
    filler = lambda: np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=int(rng.integers(5, 60)))].tobytes()  # noqa: E731
    contig, where = bytearray(filler()), {}
    for k in order:
        p = gref.revcomp(pieces[k]) if strands[k] else pieces[k]
        where[k] = len(contig)
        contig += p
        contig += filler()
    segs = [(contig_id, where[k] + 1, where[k] + len(pieces[k]), int(strands[k])) for k in range(len(pieces))]
    return bytes(contig), segs


# ---- the cases of tests/test_host_orf_edges.py and tests/test_gpu_orf_edges.py ----------------------------------------

#: prediction: the warp walks 512 payload positions per step (PRD_STEP), 16 per lane
PRD_STEP = 512
#: ORF calling: a warp tests 512 codons of a stretch per step (ORF_SPAN)
ORF_SPAN = 512
#: K4: 96-base windows (SIX_WIN), 144 bases per thread (SIX_BPT), tiles of 73 728 bases (SIX_TILE)
SIX_WIN, SIX_BPT, SIX_TILE = 96, 144, 73728
#: the check walks the nucleotide text in 32 KB tiles (MG_NUC_TILE)
NUC_TILE = 32768
#: the winner of the min_aa group of predict_payloads: the calls run at min_aa W_MIN and W_MIN + 1
W_MIN = 211


def _starts_to_plant(which):
    return ("ATG",) if which == SENSE else tuple(which)


def predict_payloads(code, which, rng):
    """[(name, Strand, cuts)] of A/C payloads with planted ORFs at the prediction scan's lane and step edges; cuts are the
    payload offsets where the multi-segment copy of the record is split (start and stop codons cut 1+2 and 2+1)."""
    sp = _starts_to_plant(which)
    out = []

    def S(n):
        return Strand(n, rng, code, SENSE if which == SENSE else tuple(which))

    def cut_codon(p):
        return [p + 1, p + 2 + 3 * 7] if p % 2 else [p + 2, p + 1 + 3 * 7]

    k = 0
    for lo in (0, 1, 2, 15, 16, 17) + tuple(range(509, 515)) + tuple(range(1021, 1027)):   # starts at lane and step edges
        n_aa = 200 + lo % 7
        s = S(lo + 3 * n_aa + 800).orf(lo, n_aa, sp[k % len(sp)], clean_stop(code, k=k))
        s.orf(lo + 301, 150, sp[(k + 1) % len(sp)], clean_stop(code, k=k + 1))          # a shorter ORF in another frame
        out.append(("start@%d" % lo, s, cut_codon(lo) + cut_codon(lo + 3 * n_aa)))
        k += 1
    for j in (1, 2):                                    # stops that straddle a lane and a step
        for r in range(PRD_STEP - 4, PRD_STEP + 4):
            x = PRD_STEP * j + r
            n_aa = 150 + j
            s = S(x + 400).orf(x - 3 * n_aa, n_aa, sp[k % len(sp)], clean_stop(code, k=k))
            out.append(("stop@%d" % x, s, cut_codon(x)))
            k += 1
    for steps in (1, 2, 3, 10):                         # ORFs over 1, 2, 3 and 10 steps: the open start carried unchanged
        n_aa = (PRD_STEP * steps - 30) // 3
        s = S(3 * n_aa + 80).orf(13, n_aa, sp[k % len(sp)], clean_stop(code, k=k))
        out.append(("steps%d" % steps, s, cut_codon(13 + 3 * n_aa)))
        k += 1
    for kk in (1, 2, 3):                                # lengths 512k + {-1, 0, 1, 2}: ORFs open at the 3' end in every frame
        for d in (-1, 0, 1, 2):
            n = PRD_STEP * kk + d
            s = S(n)
            for f, lo in enumerate((30, 37, 44)):
                s.plant(lo, sp[f % len(sp)])
            last = n - 3 - (kk % 3)
            s.plant(last, clean_stop(code, k=k))
            out.append(("len%d" % n, s, [n // 2]))
            k += 1
    for name, los, W in (("tie2-lane", (100, 104), 150), ("tie3-lane", (100, 104, 108), 150),
                         ("tie2-lanes", (100, 137), 150), ("tie3-lanes", (100, 137, 171), 200),
                         ("tie2-steps", (PRD_STEP - 3 * 160 - 2, PRD_STEP - 3 * 160 + 2), 160),
                         ("tie3-steps", (2 * PRD_STEP - 3 * 300 - 5, 2 * PRD_STEP - 3 * 300 - 1, 2 * PRD_STEP - 3 * 300 + 3), 300)):
        s = S(max(los) + 3 * W + 200)
        for i, lo in enumerate(los):                    # equal n_aa in two or three frames: the smaller lo wins
            s.orf(lo, W, sp[i % len(sp)], clean_stop(code, k=i))
        out.append((name, s, cut_codon(los[-1])))
    W = W_MIN                                           # a 5' partial and a 3' partial that tie with the best complete ORF
    s = S(3 * W + 400).orf(40, W, sp[0])
    s.plant(3 * W, clean_stop(code, k=1))              # frame 0 from codon 0: W residues, no start before its stop
    s.plant(31, clean_stop(code, k=2))                 # frame 1 from codon 1: 10 residues
    out.append(("tie-5partial", s, []))
    n = 400 + 3 * W + 2                                 # open to the last complete codon of frame 2: W residues (a 3' partial
    s = S(n).orf(40, W, sp[0])                          # ends after the complete ORF it ties with, so its start is larger)
    s.plant(2 + 3 * ((n - 2) // 3) - 3 * W, sp[-1])
    out.append(("tie-3partial", s, [n - 5]))
    for d in (0, 1, 2):                                 # min_aa at and above the winner
        s = S(6 * W + 300 + d).orf(50 + d, W, sp[d % len(sp)], clean_stop(code, k=d))
        s.orf(50 + d + 3 * W + 30, W - 20, sp[0], clean_stop(code))
        out.append(("min_aa%d" % d, s, cut_codon(50 + d)))
    s = S(3000).orf(100, 600, sp[0], clean_stop(code))  # N inside the ORF: an N codon is no stop
    s.n_run(1000, 1013)
    out.append(("n-run", s, [999, 1014]))
    return out


def call_contigs(code, which, rng):
    """[(name, Strand)] of C/G contigs (clean on both strands) with ORFs planted at the ORF caller's step edges, stretches of
    512k codons, stops on every phase's last codon and at the true-phase offsets the scan never flags (plus offset 1, minus
    offset L - 4: DESIGN section 4)."""
    sp = _starts_to_plant(which)
    st = SENSE if which == SENSE else tuple(which)
    out = []

    def S(n):
        return Strand(n, rng, code, st, alphabet=b"CG", both=True)

    for i, kc in enumerate((0, 1, 15, 16, 511, 512, 513, 1023, 1024)):   # the first start at codon kc of its stretch
        minus = bool(i % 2)
        s0 = 30 + i % 3
        x = s0 + 3 + 3 * kc
        s = S(x + 3 * 700 + 50)
        s.plant(s0, clean_stop(code, b"CG", True, i), minus)
        s.plant(x, sp[i % len(sp)], minus)
        s.plant(x + 3 * 20, sp[(i + 1) % len(sp)], minus)                  # later starts of the same stretch
        s.plant(x + 3 * 600, sp[i % len(sp)], minus)
        s.plant(x + 3 * 650, clean_stop(code, b"CG", True, i + 1), minus)
        out.append(("first-start@%d" % kc, s))
    for kk in (1, 2):                                  # stretches of exactly 512k codons
        for minus in (False, True):
            s = S(3 * ORF_SPAN * kk + 100)
            s.plant(20, clean_stop(code, b"CG", True, kk), minus)
            s.plant(23 + 3 * ORF_SPAN * kk, clean_stop(code, b"CG", True), minus)
            s.plant(23 + 3 * (ORF_SPAN * kk - (200 if minus else 2)), sp[0], minus)     # the last step's last lane on '+'

            out.append(("stretch%d" % (ORF_SPAN * kk), s))
    for L in (900, 901, 902):                          # ORFs that end on the last codon of every phase, both strands
        for p in range(3):
            last = p + 3 * ((L - p) // 3 - 1)
            s = S(L)
            s.orf(last - 3 * 250, 250, sp[p % len(sp)], clean_stop(code, b"CG", True, p), minus=bool(p % 2))
            s.orf(last - 3 * 180, 180, sp[0], clean_stop(code, b"CG", True), minus=not p % 2)
            out.append(("last-codon-L%d-p%d" % (L, p), s))
    for L in (700, 701, 702):                          # DESIGN section 4: a stop at plus offset 1 / minus offset L - 4, then a start
        s = S(L)
        s.plant(1, clean_stop(code, b"CG", True), False).orf(1 + 3 * 5, 120, sp[0], clean_stop(code, b"CG", True, 1))
        s.plant(1, clean_stop(code, b"CG", True, 2), True).orf(1 + 3 * 9, 100, sp[-1], False, True)
        out.append(("phase1-first-stop-L%d" % L, s))
    return out


def six_pairs(min_aas):
    """[(x, minus, n_res)]: two stops of one stream bounding an ORF of n_res residues (min_aa and min_aa + 1 for each min_aa),
    the lower (x = its forward position) or the higher one on the first or the last codon of a 96-base window, on a 144-base
    thread edge or on a tile edge; and pairs 47, 48 and 49 codons apart inside one thread and across two."""
    out = []
    for m in min_aas:
        for n_res in (m, m + 1):
            for E, tile in ((SIX_WIN, False), (SIX_BPT, False), (SIX_TILE, True)):
                for off in (0, E - 3, E - 2, E - 1):
                    for hi_edge in (False, True):
                        for minus in ((hi_edge,) if tile else (False, True)):      # tile edges: one strand each
                            span = 3 * (n_res + 1)
                            out.append((off - (span if hi_edge else 0), E, tile, minus, n_res))
    for gap in (47, 48, 49):
        for off in (0, 1, 2, 100):
            for minus in (False, True):
                out.append((off, SIX_BPT, False, minus, gap - 1))
    return out


def six_contigs(code, rng, min_aas, n_contig=6):
    """C/G contigs of three tiles and more with the pairs of six_pairs planted (stops only); the pairs are spread over the
    contigs and over the edges E * j + off."""
    L = 2 * SIX_TILE + 3000
    n_contig = max(n_contig, 2 + sum(1 for p in six_pairs(min_aas) if p[2]) // 2)
    strands = [Strand(L + 7 * c, rng, code, SENSE, alphabet=b"CG", both=True) for c in range(n_contig)]
    used = [[] for _ in strands]
    stop = clean_stop(code, b"CG", True)
    for i, (off, E, tile, minus, n_res) in enumerate(sorted(six_pairs(min_aas), key=lambda p: not p[2])):   # tile edges first
        span = 3 * (n_res + 1)
        js = range(0, L // E + 1)
        placed = False
        for t in range(n_contig):
            c = (i + t) % n_contig
            for j in js:
                x = E * j + off
                a, b = x - 8, x + span + 11
                if a < 0 or b > L or any(a < q and p < b for p, q in used[c]):
                    continue
                s = strands[c]
                for y in (x, x + span):
                    s.plant(s.n - y - 3 if minus else y, stop, minus)
                used[c].append((a, b))
                placed = True
                break
            if placed:
                break
        assert placed, (off, E, minus, n_res)
    return strands


def check_records(code, rng, framing):
    """[(Strand, cuts, stops)] of long A/C CDS payloads (ATG ... stop) of 2-4 text tiles, with in-frame stops whose first base
    lies at text position 32768 k - {0, 1, 2, 3} when the records are laid out one after the other in this order, each as
    pre + payload + suf with pre = len(">r%d\\n") and suf = 1 under framing (tests/test_gpu_check._table), none without."""
    out, text = [], 0
    stops = stops_of(code)
    for r, spec in enumerate(((), (0,), (1,), (2,), (3,), (0, 1, 2, 3), (3, 2), (1,))):
        n = 3 * (NUC_TILE * max(2 + r % 3, 2 * len(spec) + 2) // 3) + 3
        pre = len(b">r%d\n" % r) if framing else 0
        t0 = text + pre
        s = Strand(n, rng, code, SENSE).plant(0, "ATG").plant(n - 3, stops[r % len(stops)])   # the check reads no other start
        want = []
        for d in spec:                                 # a stop at text position 32768 k - d, in frame
            p = next(p for p in (NUC_TILE * k - d - t0 for k in range(t0 // NUC_TILE + 1, (t0 + n) // NUC_TILE + 1))
                     if 3 <= p < n - 6 and p % 3 == 0 and p // 3 not in want)
            s.plant(p, stops[(r + d) % len(stops)])
            want.append(p // 3)
        cuts = [] if r % 2 == 0 else [n // 3 + 1, 2 * n // 3 + 2, n - 2]
        out.append((s, cuts, want))
        text += pre + n + (1 if framing else 0)
    return out


def table(segs, phase=None):
    """The columns of a RecordTable that the references read, from [[(contig, start, end, strand)] per record]."""
    from types import SimpleNamespace
    rec_off = np.concatenate(([0], np.cumsum([len(r) for r in segs]))).astype(np.int64)
    flat = [x for r in segs for x in r]
    cols = [np.array([x[k] for x in flat], dtype=t) for k, t in enumerate((np.int32, np.int64, np.int64, np.int8))]
    return SimpleNamespace(rec_seg_off=rec_off, seg_contig=cols[0], seg_start=cols[1], seg_end=cols[2], seg_strand=cols[3],
                           n_rec=len(segs), n_seg=len(flat), rec_phase=None if phase is None else np.asarray(phase, np.int8))


def predict_genome(code, which, rng):
    """(contigs, segs per record, payload per record) of predict_payloads: every payload as one '+' segment, split on '+'
    and split on '-' (a third of them in mixed case)."""
    contigs, segs, pays = [], [], []
    for i, (_, s, cuts) in enumerate(predict_payloads(code, which, rng)):
        S = s.seq(rng if i % 3 == 1 else None)
        for k, minus in enumerate((False, False, True)):
            c, sg = split(S, [] if k == 0 else cuts, minus, rng, len(contigs))
            contigs.append(c)
            segs.append(sg)
            pays.append(S)
    return contigs, segs, pays


def random_contigs(rng, n=6):
    """Contigs of random A/C/G/T (some lower case, N runs) for the cross-finder checks."""
    out = []
    for k in range(n):
        a = np.frombuffer(b"ACGTACGTacgtN", dtype=np.uint8)[rng.integers(0, 13 if k % 2 else 8, size=int(rng.integers(3000, 20000)))]
        out.append(a.tobytes())
    return out
