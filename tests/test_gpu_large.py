"""The device paths on a genome past 2^32 bases with contigs of 2^31 bases or more, against references computed from a host
copy of the bytes (the library's own fetch is never the reference).

One genome of four contigs, built once for the module:

    A  3 000 017 bases        first in the forward plane; its reverse complement lies past plane index 2^33
    B  2^31 + 2^21 + 7        contig offsets past 2^31; plane index 2^31 falls inside it
    C  2^31 - 2^20 + 3        the longest contig the ORF scan takes; plane index 2^32 falls inside it
    D  1 000 003              forward-plane base past 2^32

Every ingest path packs one of them: B from host chunks (DeviceGenome.pack), C from a raw FASTA body with LF and CRLF line
ends (K0f), A and D from device memory.  The tests cover fetch on both strands, plan texts that pass byte offsets 2^31 and
2^32 in every K1 / emit variant, segments of 2^31 - 1 .. 2^31 + 1 bases, the int32 limits of a record's protein and of the
ORF scan, the host text path, K4 past plane 2^32, and (last, since they change the genome) masks and AT flags.

The module needs about 36 GB of device memory and 24 GB of host memory, and skips with both numbers when either is not free.
"""
import ctypes
import os
import resource
import time

import numpy as np
import pytest

import coracle
import genome_model
import orfcall_ref

pytestmark = pytest.mark.gpu

LENS = [3_000_017, 2**31 + 2**21 + 7, 2**31 - 2**20 + 3, 1_000_003]
A, B, C, D = range(4)
FRONT_PAD = 64                                # MG_FRONT_PAD; contigs start on multiples of 32 bases after it
NEED_DEVICE = 36 << 30
NEED_HOST = 24 << 30
POISON = 0xA5


def _layout(lens):
    base, out = FRONT_PAD, []
    for L in lens:
        out.append(base)
        base += (L + 31) // 32 * 32
    return out, base


BASES, T = _layout(LENS)
B_X31 = 2**31                                 # contig offset 2^31 in B
B_P31 = 2**31 - BASES[B]                      # offset in B of forward-plane index 2^31
C_X32 = 2**32 - BASES[C]                      # offset in C of forward-plane index 2^32
B_R33 = 2 * T - 2**33 - 1 - BASES[B]          # offset in B whose reverse-plane index is 2^33
REC_MAX = 3 * (2**31 - 1) + 2                 # longest record payload: its protein length is an int32

_ALPHA = np.frombuffer(b"ACGT" * 52 + b"acgt" * 8 + b"N" * 8 + b"nn-RYKMA", dtype=np.uint8)   # 256 entries
_EXC = np.frombuffer(b"SWBDHVxz*", dtype=np.uint8)                                        # outside the packed alphabet
_ACGT = np.zeros(256, dtype=bool)
_ACGT[np.frombuffer(b"ACGTacgt", dtype=np.uint8)] = True


def _round32(n):
    return (n + 31) // 32 * 32


def _revcomp(a):
    return np.frombuffer(coracle.revcomp(np.ascontiguousarray(a).tobytes()), dtype=np.uint8)


def _plant(t, x, exc_pos, torch):
    """N run, lower-case run, a start codon and exception bytes within a few bases of offset x of device tensor t."""
    def put(lo, b):
        t[lo:lo + len(b)] = torch.tensor(np.frombuffer(b, dtype=np.uint8).copy(), device=t.device)
    put(x - 120, b"N" * 40)
    put(x + 40, b"acgtn" * 8)
    put(x - 50, b"ATGATG")
    put(x - 7, b"S-W-B-zDHVx*")
    exc_pos += [x - 7, x - 5, x - 3, x - 1, x, x + 1, x + 2, x + 3, x + 4]


def _draw(torch, gen, n, x_list):
    """n random bytes over the alphabet on the device, 3000 scattered exception bytes, and planted runs near each x."""
    lut = torch.tensor(_ALPHA.copy(), device="cuda")
    t = torch.empty(n, dtype=torch.uint8, device="cuda")
    step = 1 << 26
    for a in range(0, n, step):
        b = min(n, a + step)
        t[a:b] = lut[torch.randint(0, 256, (b - a,), generator=gen, device="cuda", dtype=torch.uint8).long()]
    pos = torch.randint(0, n, (3000,), generator=gen, device="cuda")
    exc = torch.tensor(_EXC.copy(), device="cuda")
    t[pos] = exc[torch.randint(0, _EXC.size, (3000,), generator=gen, device="cuda")]
    planted = []
    for x in x_list:
        _plant(t, x, planted, torch)
    return t, pos.cpu().numpy(), planted


def _fasta_body(seq):
    """seq as a FASTA body of 60-column lines: LF line ends in the first half, CRLF in the second."""
    n = seq.size
    half = (n // 2) // 60 * 60
    m1, m2 = half // 60, (n - half) // 60
    tail = n - half - 60 * m2
    raw = np.empty(m1 * 61 + m2 * 62 + (tail + 2 if tail else 0), dtype=np.uint8)
    v1 = raw[:m1 * 61].reshape(m1, 61)
    v1[:, :60] = seq[:half].reshape(m1, 60)
    v1[:, 60] = 10
    v2 = raw[m1 * 61:m1 * 61 + m2 * 62].reshape(m2, 62)
    v2[:, :60] = seq[half:half + 60 * m2].reshape(m2, 60)
    v2[:, 60] = 13
    v2[:, 61] = 10
    if tail:
        raw[-tail - 2:-2] = seq[n - tail:]
        raw[-2:] = (13, 10)
    return raw


class Big(object):
    pass


@pytest.fixture(scope="module")
def big():
    import torch
    from magot_b200 import engine
    free, total = torch.cuda.mem_get_info()
    if free < NEED_DEVICE:
        pytest.skip("needs %d bytes of free device memory, %d are free" % (NEED_DEVICE, free))
    host_free = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    if host_free < NEED_HOST:
        pytest.skip("needs %d bytes of free host memory, %d are free" % (NEED_HOST, host_free))
    t0 = time.time()
    s = Big()
    s.used0 = total - free
    s.dev_peak = 0
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2024)
    offs = np.concatenate(([0], np.cumsum(LENS)))
    s.host = np.empty(int(offs[-1]), dtype=np.uint8)
    s.hv = [s.host[offs[c]:offs[c + 1]] for c in range(4)]
    s.exc = {}
    g = engine.DeviceGenome(LENS, device=0)
    crossings = {A: [LENS[A] - 200], B: [B_X31, B_P31, B_R33], C: [C_X32], D: [500_000]}
    for c in (A, B, C, D):
        t, pos, planted = _draw(torch, gen, LENS[c], crossings[c])
        torch.from_numpy(s.hv[c]).copy_(t)
        s.exc[c] = sorted(set(int(p) for p in pos[:20]) | set(planted))
        if c == B:
            g.pack(B, s.hv[B])                        # 64 MiB host chunks at offsets up to past 2^31
        elif c == C:
            raw = _fasta_body(s.hv[C])
            assert raw.size > 2**31
            g.pack_fasta(C, raw)                      # K0f over more than 2^31 raw bytes
            del raw
        else:
            g.pack_device(c, t.data_ptr(), LENS[c])
        torch.cuda.synchronize()
        del t
    torch.cuda.empty_cache()
    g.finalize()
    s.g = g
    s.t_build = time.time() - t0
    yield s
    g.close()
    print("\n[test_gpu_large] genome built in %.1f s; device memory used by the module, at most %.1f GB (sampled after each "
          "test); host peak RSS %.1f GB" % (s.t_build, s.dev_peak / 1e9,
                                            resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6))


@pytest.fixture(autouse=True)
def _sample_memory(big):
    import torch
    yield
    free, total = torch.cuda.mem_get_info()
    big.dev_peak = max(big.dev_peak, total - free - big.used0)


@pytest.fixture()
def tune():
    from magot_b200 import _lib

    def set_(key, v):
        _lib.check(_lib.lib.mg_tune(key.encode(), v))
    yield set_
    set_("emit", 0)
    set_("k1", 0)
    set_("six", 2)


def test_layout():
    """The crossings the module is built around, under the documented layout: if the layout changes, this fails."""
    assert BASES[B] < 2**31 < BASES[B] + LENS[B]
    assert 0 < B_P31 < LENS[B] and B_X31 < LENS[B]
    assert BASES[C] <= 2**32 < BASES[C] + LENS[C] and C_X32 == 2_142_386_368
    assert BASES[D] > 2**32
    assert 2 * T - BASES[A] - LENS[A] > 2**33           # A's reverse complement
    assert 0 < B_R33 < LENS[B]
    assert LENS[C] < 2**31 <= LENS[B]


# ---- 1. fetch -------------------------------------------------------------------------------------------------------------

def test_fetch_across_boundaries(big):
    wins = [(B, B_X31 - 5000, B_X31 + 5000), (B, B_P31 - 3000, B_P31 + 3000), (C, C_X32 - 5000, C_X32 + 5000),
            (B, B_R33 - 3000, B_R33 + 3000)]
    for c in range(4):
        wins += [(c, 0, 100), (c, LENS[c] - 100, LENS[c])]
        wins += [(c, max(0, p - 50), min(LENS[c], p + 50)) for p in big.exc[c]]
    for c, lo, hi in wins:
        want = big.hv[c][lo:hi]
        assert big.g.fetch(c, lo, hi) == want.tobytes(), (c, lo, hi)
        assert big.g.fetch(c, lo, hi, minus=True) == _revcomp(want).tobytes(), (c, lo, hi, "-")


# ---- 2. plan texts ---------------------------------------------------------------------------------------------------------

def _clamp(c, a, b):
    """contig[a-1:b] with Python slice rules: (lo, hi)."""
    L = LENS[c]
    i, k = a - 1, b
    i = max(i + L, 0) if i < 0 else min(i, L)
    k = max(k + L, 0) if k < 0 else min(k, L)
    return i, max(i, k)


def _table(recs, rng, framing=True):
    from magot_b200 import engine
    rec_off, cid, st, en, sd = [0], [], [], [], []
    for r in recs:
        for (c, a, b, m) in r:
            cid.append(c); st.append(a); en.append(b); sd.append(m)
        rec_off.append(len(cid))
    R = len(recs)
    pre = rng.integers(0, 7, size=R).astype(np.int32) if framing else np.zeros(R, np.int32)
    suf = rng.integers(0, 3, size=R).astype(np.int32) if framing else np.zeros(R, np.int32)
    lit_off = np.concatenate([[0], np.cumsum(pre.astype(np.int64) + suf)])[:R].astype(np.int64)
    lit = rng.integers(65, 91, size=int(pre.sum() + suf.sum())).astype(np.uint8)
    return engine.RecordTable(rec_off, cid, st, en, sd, lit_off, pre, suf, lit)


def _frame(body, body_off, tbl, lead=None):
    """prefix + ('X' where lead) + body[r] + suffix of every record, spliced by the C oracle (contig 0 = body, 1 = the
    literals, 2 = "X")."""
    R = tbl.n_rec
    pre_lo = tbl.rec_lit_off
    pre_hi = pre_lo + tbl.rec_pre_len
    lo = np.stack([pre_lo, np.zeros(R, np.int64), body_off[:-1], pre_hi], axis=1)
    hi = np.stack([pre_hi, np.zeros(R, np.int64) if lead is None else lead.astype(np.int64), body_off[1:],
                   pre_hi + tbl.rec_suf_len], axis=1)
    cid = np.tile(np.array([1, 2, 0, 1], np.int32), R)
    lit = tbl.lit if tbl.lit.size else np.zeros(1, np.uint8)
    text, _ = coracle.splice([body if body.size else np.zeros(1, np.uint8), lit, b"X"], np.arange(R + 1) * 4, cid,
                             lo.ravel(), hi.ravel(), np.zeros(4 * R, np.int8))
    return text


def _reference(big, recs, tbl):
    """(nucleotide text, protein text with trimX, without, nuc lengths, aa lengths with trimX, without) from the host copy:
    Python-clamped intervals spliced and translated by the C oracle.  Built in this order so that at most one text of the
    size of the nucleotide text is on the host at a time."""
    cid, lo, hi, mi = [], [], [], []
    for r in recs:
        for (c, a, b, m) in r:
            i, k = _clamp(c, a, b)
            cid.append(c); lo.append(i); hi.append(k); mi.append(m)
    nuc, off = coracle.splice(big.hv, tbl.rec_seg_off, cid, lo, hi, mi)
    aa, aa_off, aa_len = coracle.splice_translate(nuc, off)
    nl = np.diff(off)
    first = np.zeros(tbl.n_rec, dtype=bool)             # the first codon holds a base outside ACGT: trimX dropped an 'X'
    has = nl >= 3
    idx = off[:-1][has]
    first[has] = ~_ACGT[nuc[idx[:, None] + np.arange(3)]].all(axis=1)
    del nuc
    lead = first & (aa_len >= 0)
    text_p1 = _frame(aa, aa_off, tbl)
    text_p0 = _frame(aa, aa_off, tbl, lead)
    del aa
    # the framed nucleotide text in one splice: the literals are a fifth contig
    fcid, flo, fhi, fmi, fo = [], [], [], [], [0]
    e = 0
    for r in range(tbl.n_rec):
        p0 = int(tbl.rec_lit_off[r])
        p1 = p0 + int(tbl.rec_pre_len[r])
        n = int(tbl.rec_seg_off[r + 1] - tbl.rec_seg_off[r])
        fcid += [4] + cid[e:e + n] + [4]
        flo += [p0] + lo[e:e + n] + [p1]
        fhi += [p1] + hi[e:e + n] + [p1 + int(tbl.rec_suf_len[r])]
        fmi += [0] + mi[e:e + n] + [0]
        fo.append(len(fcid))
        e += n
    lit = tbl.lit if tbl.lit.size else np.zeros(1, np.uint8)
    text_n, _ = coracle.splice(big.hv + [lit], fo, fcid, flo, fhi, fmi)
    return text_n, text_p1, text_p0, nl, aa_len, np.where(aa_len >= 0, aa_len + lead, aa_len)


def _small_recs(rng, n):
    centres = [(B, B_X31), (B, B_P31), (C, C_X32), (B, B_R33), (A, LENS[A]), (B, 1), (C, LENS[C]), (D, LENS[D]), (D, 1),
               (B, LENS[B]), (A, 1)]
    recs = []
    for _ in range(n):
        r = []
        for _ in range(int(rng.integers(0, 8))):
            c, x = centres[int(rng.integers(0, len(centres)))]
            m = int(rng.integers(0, 2))
            kind = rng.random()
            if kind < 0.8:
                a = x + int(rng.integers(-300, 300))
                r.append((c, a, a + int(rng.integers(-1, 200)), m))
            elif kind < 0.9:
                r.append((c, LENS[c] + 5, LENS[c] + 50, m))
            else:
                r.append((c, -int(rng.integers(1, 400)), -1, m))
        recs.append(r)
    return recs


def _big_recs():
    s = 7_777
    return [[(B, 1, LENS[B], 0)],
            [(B, 1, LENS[B], 1)],
            [(B, -(2**31 + 100), -1, 1)],
            [(A, 1001, 2_000_000, 0), (B, s, s + 2**31, 1), (C, C_X32 - 499_999, C_X32 + 500_000, 0), (D, 1, LENS[D], 1)]]


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check_out(torch, out, ref, total):
    assert torch.equal(out[:total], ref)
    tail = out[_round32(total):]
    assert tail.numel() > 0 and bool((tail == POISON).all())


def test_plan_texts_past_2_32(big, tune):
    """A few thousand small records near the crossings with four records of 2^31 bases or more among them (B whole on both
    strands, B through negative coordinates, one multi-segment record): both texts, lengths and totals in every K1 / emit
    variant, through prepare and prepare_async with a deferred record pass, K23 and the one-launch products."""
    import torch
    from magot_b200 import engine, _lib
    rng = np.random.default_rng(31)
    small = _small_recs(rng, 3000)
    recs = small[:1000] + _big_recs()[:2] + small[1000:2000] + _big_recs()[2:] + small[2000:]
    tbl = _table(recs, rng)
    text_n, text_p1, text_p0, nl, al1, al0 = _reference(big, recs, tbl)
    tot_n, tot_p1, tot_p0 = text_n.size, text_p1.size, text_p0.size
    assert tot_n > 2**33 and (nl >= 2**31).sum() == 4
    ref_n = _dev(torch, text_n)
    del text_n
    ref_p = {True: _dev(torch, text_p1), False: _dev(torch, text_p0)}
    tot_p = {True: tot_p1, False: tot_p0}
    al = {True: al1, False: al0}
    del text_p1, text_p0
    out_n = torch.empty(_round32(tot_n) + 64, dtype=torch.uint8, device="cuda")
    out_p = torch.empty(_round32(max(tot_p1, tot_p0)) + 64, dtype=torch.uint8, device="cuda")

    srecs = small[:200]                                 # the second plan of the one-launch products
    stbl = _table(srecs, rng)
    s_n, s_p, _, _, _, _ = _reference(big, srecs, stbl)
    sref_n, sref_p = _dev(torch, s_n), _dev(torch, s_p)
    sout_n = torch.empty(_round32(s_n.size) + 64, dtype=torch.uint8, device="cuda")
    sout_p = torch.empty(_round32(s_p.size) + 64, dtype=torch.uint8, device="cuda")

    plan = engine.Plan(big.g, tbl)
    splan = engine.Plan(big.g, stbl)
    try:
        for emit in (0, 1, 2):
            for k1 in (0, 1):
                tune("emit", emit)
                tune("k1", k1)
                where = (emit, k1)
                for trimx in (True, False):
                    assert plan.prepare(trimx=trimx) == (tot_n, tot_p[trimx]), where
                    n_len, a_len = plan.lengths()
                    assert np.array_equal(n_len, nl) and np.array_equal(a_len, al[trimx]), where
                    out_n.fill_(POISON)
                    out_p.fill_(POISON)
                    plan.emit_device(out_n.data_ptr(), protein=False)
                    plan.emit_device(out_p.data_ptr(), protein=True)
                    torch.cuda.synchronize()
                    _check_out(torch, out_n, ref_n, tot_n)
                    _check_out(torch, out_p, ref_p[trimx], tot_p[trimx])

                    plan.prepare_async(tot_n, tot_p[trimx], trimx=trimx, defer_records=True)
                    out_n.fill_(POISON)
                    out_p.fill_(POISON)
                    plan.emit_device(out_n.data_ptr(), protein=False)
                    # the one-launch K1 runs the record pass inside the piece pass: nothing is deferred
                    assert plan.totals() == (tot_n, tot_p[trimx] if k1 else 0), where
                    plan.prepare_prot()
                    plan.emit_device(out_p.data_ptr(), protein=True)
                    assert plan.totals() == (tot_n, tot_p[trimx]), where
                    n_len, a_len = plan.lengths()
                    assert np.array_equal(n_len, nl) and np.array_equal(a_len, al[trimx]), where
                    torch.cuda.synchronize()
                    _check_out(torch, out_n, ref_n, tot_n)
                    _check_out(torch, out_p, ref_p[trimx], tot_p[trimx])

                plan.prepare()                           # K23, then the products with the small plan on either side
                splan.prepare()
                out_n.fill_(POISON)
                out_p.fill_(POISON)
                _lib.check(_lib.lib.mg_emit_nuc_prot_device(plan.handle, out_n.data_ptr(), out_p.data_ptr(), None))
                torch.cuda.synchronize()
                _check_out(torch, out_n, ref_n, tot_n)
                _check_out(torch, out_p, ref_p[True], tot_p1)
                for big_first in (True, False):
                    for t in (out_n, out_p, sout_n, sout_p):
                        t.fill_(POISON)
                    if big_first:
                        _lib.check(_lib.lib.mg_emit_products_device(plan.handle, out_n.data_ptr(), splan.handle,
                                                                    sout_n.data_ptr(), sout_p.data_ptr(), None))
                    else:
                        _lib.check(_lib.lib.mg_emit_products_device(splan.handle, sout_n.data_ptr(), plan.handle,
                                                                    out_n.data_ptr(), out_p.data_ptr(), None))
                    torch.cuda.synchronize()
                    _check_out(torch, out_n, ref_n, tot_n)
                    _check_out(torch, sout_n, sref_n, s_n.size)
                    _check_out(torch, sout_p if big_first else out_p, sref_p if big_first else ref_p[True],
                               s_p.size if big_first else tot_p1)
    finally:
        plan.close()
        splan.close()
        del out_n, out_p, ref_n, ref_p
        torch.cuda.empty_cache()


# ---- 3. segments of 2^31 - 1, 2^31 and 2^31 + 1 bases --------------------------------------------------------------------

@pytest.mark.parametrize("minus", [0, 1])
def test_segment_lengths_around_2_31(big, minus):
    import torch
    from magot_b200 import engine
    rng = np.random.default_rng(3)
    out = torch.empty(_round32(2**31 + 1) + 64, dtype=torch.uint8, device="cuda")
    K = 4096
    try:
        for j, n in enumerate((2**31 - 1, 2**31, 2**31 + 1)):
            lo = 1001 + 2 * j + 6 * minus                 # odd offsets of B
            tbl = _table([[(B, lo + 1, lo + n, minus)]], rng, framing=False)
            plan = engine.Plan(big.g, tbl)
            try:
                assert plan.prepare()[0] == n, n
                n_len, _ = plan.lengths()
                assert int(n_len[0]) == n
                plan.emit_device(out.data_ptr(), protein=False)
                torch.cuda.synchronize()
                head = out[:K].cpu().numpy()
                tail = out[n - K:n].cpu().numpy()
            finally:
                plan.close()
            seq = big.hv[B]
            if minus:
                want_head, want_tail = _revcomp(seq[lo + n - K:lo + n]), _revcomp(seq[lo:lo + K])
            else:
                want_head, want_tail = seq[lo:lo + K], seq[lo + n - K:lo + n]
            assert np.array_equal(head, want_head), (n, "head")
            assert np.array_equal(tail, want_tail), (n, "tail")
    finally:
        del out
        torch.cuda.empty_cache()


# ---- 4. the int32 limits --------------------------------------------------------------------------------------------------

def test_record_protein_limit(big):
    """A record of exactly 3 * (2^31 - 1) + 2 bases (three segments of B and C) is planned with 2^31 - 1 amino acids; one base
    more is refused when the plan is created."""
    from magot_b200 import engine, _lib
    rng = np.random.default_rng(4)
    rest = REC_MAX - LENS[B] - LENS[C]
    assert 0 < rest < LENS[B]
    segs = [(B, 1, LENS[B], 0), (C, 1, LENS[C], 1), (B, 11, 10 + rest, 0)]
    plan = engine.Plan(big.g, _table([segs], rng, framing=False))
    try:
        assert plan.prepare(trimx=False) == (REC_MAX, 2**31 - 1)
        n_len, a_len = plan.lengths()
        assert (int(n_len[0]), int(a_len[0])) == (REC_MAX, 2**31 - 1)
    finally:
        plan.close()
    segs[2] = (B, 11, 11 + rest, 0)
    with pytest.raises(_lib.MagotError, match=r"limited to 3 \* \(2\^31 - 1\) \+ 2"):
        engine.Plan(big.g, _table([segs], rng, framing=False))


def test_orf_scans_refuse_contigs_of_2_31(big):
    from magot_b200 import orfs, _lib
    with pytest.raises(_lib.MagotError, match=r"2\^31 bases"):
        orfs.sixframe_list(big.g, [B], 30)
    recs, aa = orfs.sixframe_list(big.g, [D], 30)
    assert recs.size > 0 and len(aa) == int(recs["len"].sum())
    with pytest.raises(_lib.MagotError, match=r"2\^31 bases"):
        orfs.call_orfs(big.g, [B], 30)
    recs, aa = orfs.call_orfs(big.g, [D], 30)
    assert recs.size > 0 and len(aa) == int(recs["len"].sum())


# ---- 5. the host text path -------------------------------------------------------------------------------------------------

def test_run_table_bytes_past_2_31(big):
    from magot_b200 import engine
    tbl = _table([[(B, 1, LENS[B], 0)]], np.random.default_rng(5), framing=False)
    text, lens = engine.run_table(big.g, tbl, want_lengths=True)
    n = len(text)
    assert isinstance(text, bytes) and n == LENS[B] > 2**31
    assert int(lens[0][0]) == LENS[B]
    assert np.array_equal(np.frombuffer(text, dtype=np.uint8), big.hv[B])


# ---- 6. K4 past plane 2^32 -------------------------------------------------------------------------------------------------

def _six_want(big, ids, min_aa):
    aa, rows = [], []
    for c in ids:
        a, r = coracle.sixframe(big.hv[c], min_aa)
        aa.append(a)
        rows.append(np.concatenate([np.full((len(r), 1), c, np.int64), r.reshape(-1, 4)], axis=1))
    return b"".join(aa), np.concatenate(rows)


def _six_got(recs):
    return np.stack([recs[f].astype(np.int64) for f in ("contig", "frame", "minus", "start", "len")], axis=1)


def test_sixframe_past_2_32(big, tune):
    from magot_b200 import orfs
    for ids in ([D], [A, D]):
        for min_aa in (0, 30):
            want_aa, want_rows = _six_want(big, ids, min_aa)
            recs, aa = orfs.sixframe_list(big.g, ids, min_aa)
            assert aa == want_aa and np.array_equal(_six_got(recs), want_rows), (ids, min_aa)
    want_aa, want_rows = _six_want(big, [C], 100)
    assert len(want_rows) > 0
    for mode in (2, 0):
        tune("six", mode)
        recs, aa = orfs.sixframe_list(big.g, [C], 100)
        assert aa == want_aa and np.array_equal(_six_got(recs), want_rows), mode


def test_orfcall_past_2_32(big, tune):
    from magot_b200 import orfs
    contigs = [b"", b"", b"", big.hv[D].tobytes()]
    want_recs, want_aa = orfcall_ref.call_list(contigs, [D], 30)
    win = 1_000_000
    for mode in (2, 0):
        tune("six", mode)
        recs, aa = orfs.call_orfs(big.g, [D], 30)
        got = [tuple(int(v) for v in r) for r in recs[["contig", "minus", "phase", "flags", "start_codon", "lo", "hi", "len",
                                                           "aa_off"]].tolist()]
        assert got == want_recs and aa == want_aa, mode
        recs, aa = orfs.call_orfs(big.g, [C], 30)
        near = recs[(recs["lo"] >= C_X32 - win) & (recs["hi"] <= C_X32 + win)]
        assert near.size > 100 and (near["lo"] < C_X32).any() and (near["hi"] > C_X32).any()
        for r in near:
            seq = big.hv[C][int(r["lo"]):int(r["hi"])]
            if r["minus"]:
                seq = _revcomp(seq)
            prot = coracle.translate(seq[:-3].tobytes(), trimX=False)
            got = aa[int(r["aa_off"]):int(r["aa_off"]) + int(r["len"])]
            assert got == b"M" + prot[1:], (mode, int(r["lo"]), int(r["hi"]), int(r["minus"]))


# ---- 7. masks and AT flags (last: they change the genome) -----------------------------------------------------------------

def _at_flags(g, c, lo, hi):
    from magot_b200 import _lib
    out = np.full(hi - lo, 7, dtype=np.uint8)
    _lib.check(_lib.lib.mg_genome_at_flags(g.handle, c, lo, hi, ctypes.c_void_p(out.ctypes.data), None))
    return out


def test_masks_and_at_flags_past_2_32(big):
    """Soft, hard and upper_first masks across B's offset 2^31, C's plane-2^32 crossing and in D; fetch on both strands and
    AT flags over the windows against the byte model, then K2 / K3 / K23 of a plan over the masked windows, one of whose
    trimX decisions the hard mask changes."""
    import torch
    from magot_b200 import engine, _lib
    wins = [(B, B_X31 - 1024, B_X31 + 1024), (C, C_X32 - 1024, C_X32 + 1024), (D, 0, 8192)]
    assert all(lo % 8 == 0 for _, lo, _ in wins)
    model = genome_model.Genome([big.hv[c][lo:hi].tobytes() for c, lo, hi in wins])

    def mask(ivs, hard=False, upper_first=False):
        big.g.mask([c for c, _, _ in ivs], [a for _, a, _ in ivs], [b for _, _, b in ivs], hard=hard, upper_first=upper_first)
        w = {c: (k, lo) for k, (c, lo, _) in enumerate(wins)}
        model.mask([w[c][0] for c, _, _ in ivs], [a - w[c][1] for c, a, _ in ivs], [b - w[c][1] for c, _, b in ivs],
                   hard=hard, upper_first=upper_first)
        for k, (c, lo, hi) in enumerate(wins):
            for m in (False, True):
                assert big.g.fetch(c, lo, hi, minus=m) == model.fetch(k, 0, hi - lo, minus=m), (c, m, hard, upper_first)
            assert np.array_equal(_at_flags(big.g, c, lo, hi), model.at_flags(k, 0, hi - lo)), (c, hard, upper_first)

    mask([(B, B_X31 - 300, B_X31 + 300), (C, C_X32 - 200, C_X32 + 250), (D, 1000, 5000)])
    assert big.hv[B][B_X31 - 50:B_X31 - 47].tobytes() == b"ATG"
    mask([(B, B_X31 - 50, B_X31 + 60), (C, C_X32 + 10, C_X32 + 20), (D, 2000, 2100)], hard=True)
    mask([(D, 3000, 3100), (B, B_X31 + 500, B_X31 + 700)], upper_first=True)

    recs = [[(B, B_X31 - 49, B_X31 + 300, 0)],                       # starts on the hard-masked ATG: trimX drops its 'X'
            [(B, B_X31 - 700, B_X31 + 20, 1), (C, C_X32 - 600, C_X32 + 900, 0)],
            [(C, C_X32 - 30, C_X32 + 40, 1), (D, 1500, 2500, 0), (D, 2050, 3050, 1)]]
    tbl = _table(recs, np.random.default_rng(7))
    w = {c: (k, lo) for k, (c, lo, _) in enumerate(wins)}
    cid, lo, hi, mi = [], [], [], []
    for r in recs:
        for (c, a, b, m) in r:
            cid.append(w[c][0]); lo.append(a - 1 - w[c][1]); hi.append(b - w[c][1]); mi.append(m)
    nuc, off = coracle.splice([bytes(x) for x in model.contigs], tbl.rec_seg_off, cid, lo, hi, mi)
    aa, aa_off, aa_len = coracle.splice_translate(nuc, off)
    assert int(aa_len[0]) == (B_X31 + 300 - (B_X31 - 50)) // 3 - 1
    want_n, want_p = _frame(nuc, off, tbl), _frame(aa, aa_off, tbl)
    plan = engine.Plan(big.g, tbl)
    try:
        assert plan.prepare() == (want_n.size, want_p.size)
        n_len, a_len = plan.lengths()
        assert np.array_equal(n_len, np.diff(off)) and np.array_equal(a_len, aa_len)
        assert plan.emit_host(False).tobytes() == want_n.tobytes()
        assert plan.emit_host(True).tobytes() == want_p.tobytes()
        out_n = torch.full((_round32(want_n.size) + 64,), POISON, dtype=torch.uint8, device="cuda")
        out_p = torch.full((_round32(want_p.size) + 64,), POISON, dtype=torch.uint8, device="cuda")
        _lib.check(_lib.lib.mg_emit_nuc_prot_device(plan.handle, out_n.data_ptr(), out_p.data_ptr(), None))
        torch.cuda.synchronize()
        _check_out(torch, out_n, _dev(torch, want_n), want_n.size)
        _check_out(torch, out_p, _dev(torch, want_p), want_p.size)
    finally:
        plan.close()
