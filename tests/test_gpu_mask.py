"""K5 masking (mg_genome_mask, genome_tools mask_from_gff) and K6 AT flags (mg_genome_at_flags), bit-exact against the byte
model genome_model: both strands after every mask, the exception count, every start and end residue of a packed word,
intervals across the warp stride, contig ends next to the padding, sequences of masks on one genome, the regrow of the
R/Y/K/M hit list, every reader of a masked genome (K2/K3 in each variant, the six-frame scan, ORF calling, the device emit),
AT flags at any lo / hi and across the 256 MiB staging boundary, argument checks that leave the genome unchanged, and
counts / plans prepared before a genome change, whose emits must fail instead of mixing two genomes."""
import ctypes

import numpy as np
import pytest

import coracle
import gencode_ref as gref
import genome_model as gm
import orfcall_ref

pytestmark = pytest.mark.gpu

#: the packed alphabet, lower-case R/Y/K/M and bytes outside it (exceptions)
ALPHA = np.frombuffer(b"ACGTacgtNn-RYKMrykmW* \xe9", dtype=np.uint8)
#: contig lengths around the 8-base word, the 32-base contig alignment and the 256-base warp stride
LENS = (0, 1, 7, 8, 9, 31, 32, 33, 255, 256, 257, 70001)
MG_ESTATE = -4


@pytest.fixture(scope="module")
def mg():
    import magot_b200
    return magot_b200


@pytest.fixture()
def tune(mg):
    from magot_b200 import _lib
    yield lambda key, v: _lib.check(_lib.lib.mg_tune(key, v))
    for key, v in ((b"emit", 0), (b"k1", 0), (b"six", 2)):
        _lib.check(_lib.lib.mg_tune(key, v))


def _genome(contigs):
    from magot_b200 import engine
    g = engine.DeviceGenome([len(c) for c in contigs], device=0)
    for i, c in enumerate(contigs):
        g.pack(i, np.frombuffer(bytes(c), dtype=np.uint8))
    g.finalize()
    return g


def _random_contigs(rng, lens=LENS, alpha=ALPHA, p=None):
    return [alpha[rng.choice(alpha.size, size=n, p=p)].tobytes() for n in lens]


def _intervals(rng, lens):
    """(contig, lo, hi) of a table with every kind of interval on every non-empty contig: empty, one base, each start and
    end residue mod 8, nested, overlapping, duplicated, the whole contig, longer than the 256-base warp stride and than
    8192 bases, and touching either contig end."""
    out = []
    for ci, L in enumerate(lens):
        if L == 0:
            continue
        a = int(rng.integers(0, L))
        out += [(ci, a, a), (ci, a, a + 1), (ci, 0, 1), (ci, L - 1, L), (ci, L, L)]
        if rng.random() < 0.25:                      # not everywhere: bases next to interval ends must stay unmasked
            out.append((ci, 0, L))
        for s in range(8):
            for e in range(8):
                lo = 8 * int(rng.integers(0, max(1, L // 8))) + s
                hi = lo + 8 * int(rng.integers(0, 40)) + (e - s) % 8
                if hi <= L:
                    out.append((ci, lo, hi))
        b = int(rng.integers(a, L + 1))
        out += [(ci, a, b), (ci, a, b), (ci, (a + b) // 2, b), (ci, a, (a + b) // 2 + 1)]     # duplicated, nested
        c = min(L, b + int(rng.integers(0, 600)))
        out.append((ci, max(a, b - 5), c))                                                   # overlapping
        for n in (257, 300, 8193, 9000):
            if n <= L:
                lo = int(rng.integers(0, L - n + 1))
                out.append((ci, lo, lo + n))
    order = rng.permutation(len(out))
    return [out[k] for k in order]


def _cols(ivs):
    return ([x[0] for x in ivs], [x[1] for x in ivs], [x[2] for x in ivs])


def _mask(g, model, ivs, hard=False, upper_first=False):
    c, lo, hi = _cols(ivs)
    g.mask(c, lo, hi, hard=hard, upper_first=upper_first)
    model.mask(c, lo, hi, hard=hard, upper_first=upper_first)


def _check(g, model, rng, n_sub=6):
    """Both strands of every contig, whole and on random sub-slices, and the exception count, against the model."""
    for ci, c in enumerate(model.contigs):
        L = len(c)
        for minus in (False, True):
            assert g.fetch(ci, 0, L, minus) == model.fetch(ci, 0, L, minus), (ci, L, minus)
        for _ in range(n_sub):
            a = int(rng.integers(0, L + 1))
            b = int(rng.integers(a, L + 1))
            for minus in (False, True):
                assert g.fetch(ci, a, b, minus) == model.fetch(ci, a, b, minus), (ci, a, b, minus)
    assert g.finalize() == model.n_exceptions()


# ---- 1-3: masks against the model ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("hard", [False, True])
@pytest.mark.parametrize("upper_first", [False, True])
def test_mask_random(mg, hard, upper_first):
    rng = np.random.default_rng(100 + 2 * hard + upper_first)
    contigs = _random_contigs(rng) + _random_contigs(rng, lens=rng.integers(0, 3000, size=8))
    model = gm.Genome(contigs)
    g = _genome(contigs)
    try:
        _check(g, model, rng)
        _mask(g, model, _intervals(rng, [len(c) for c in contigs]), hard=hard, upper_first=upper_first)
        _check(g, model, rng)
    finally:
        g.close()


def test_mask_sequence(mg):
    """Soft, hard, soft after upper-casing, then empty tables with and without upper-casing on ONE genome: exceptions are
    lower-cased, dropped, added and de-duplicated across calls, and the two strands follow."""
    rng = np.random.default_rng(110)
    contigs = _random_contigs(rng)
    lens = [len(c) for c in contigs]
    model = gm.Genome(contigs)
    g = _genome(contigs)
    try:
        for hard, upper_first, empty in ((False, False, False), (True, False, False), (False, True, False),
                                         (False, True, True), (True, False, True), (False, False, False)):
            ivs = [] if empty else _intervals(rng, lens)[::3]
            _mask(g, model, ivs, hard=hard, upper_first=upper_first)
            _check(g, model, rng)
    finally:
        g.close()


def test_mask_iupac_regrow(mg):
    """More than 65 536 R/Y/K/M hits inside the soft intervals of one call (the first listing pass holds 65 536): the list
    is rebuilt with room for all of them; overlapping intervals list a base twice."""
    rng = np.random.default_rng(120)
    iupac = np.frombuffer(b"RYKMRYKMRYKMRYKMRYKMACGTNn", dtype=np.uint8)
    contigs = [_random_contigs(rng, lens=(1000,))[0], iupac[rng.integers(0, iupac.size, size=200_003)].tobytes(),
               _random_contigs(rng, lens=(777,))[0]]
    ivs = [(1, 8 * k * 1000 + 3, min(200_003, 8 * k * 1000 + 60_001)) for k in range(0, 25, 3)]
    ivs += [(1, 0, 200_003), (0, 10, 990), (2, 0, 777)]
    model = gm.Genome(contigs)
    hits = sum(sum(1 for x in contigs[c][a:b] if x in b"RYKM") for c, a, b in ivs)
    assert hits > 65_536 and hits > model.listed[1].size
    g = _genome(contigs)
    try:
        _mask(g, model, ivs)
        _check(g, model, rng)
        _mask(g, model, ivs[:4], upper_first=True)          # the listed bytes upper-cased, then lower-cased again in part
        _check(g, model, rng)
    finally:
        g.close()


# ---- 4: readers of a masked genome -----------------------------------------------------------------------------------------

def _plan_table(rng, contigs, hard_ivs, n_rec=300):
    """Random records with '+' and '-' segments (coordinates off either end, Python slice rules) over `contigs`; every
    third record starts where a hard interval starts ('+') or ends where one ends ('-'), so that its first codon is masked."""
    from magot_b200 import engine
    segs = []
    for r in range(n_rec):
        row = []
        if r % 3 == 0 and hard_ivs:
            c, a, b = hard_ivs[int(rng.integers(0, len(hard_ivs)))]
            if r % 2:
                row.append((c, a + 1, a + int(rng.integers(3, 400)), 0))
            else:
                row.append((c, max(1, b - int(rng.integers(3, 400))), b, 1))
        for _ in range(int(rng.integers(0 if row else 1, 6))):
            c = int(rng.integers(0, len(contigs)))
            L = len(contigs[c])
            a = int(rng.integers(-20, L + 20))
            row.append((c, a, a + int(rng.integers(-3, 500)), int(rng.integers(0, 2))))
        segs.append(row)
    flat = [x for row in segs for x in row]
    rec_off = np.concatenate(([0], np.cumsum([len(row) for row in segs]))).astype(np.int64)
    st = np.array([min(x[1], x[2]) for x in flat], dtype=np.int64)
    en = np.array([max(x[1], x[2]) for x in flat], dtype=np.int64)
    z = np.zeros(n_rec, dtype=np.int32)
    tbl = engine.RecordTable(rec_off, [x[0] for x in flat], st, en, [x[3] for x in flat], np.zeros(n_rec, np.int64), z, z,
                             np.zeros(0, np.uint8))
    return tbl


def _plan_want(tbl, contigs):
    """Spliced text, protein text and per-record lengths of the C oracle on the model's bytes."""
    lens = np.array([len(c) for c in contigs], dtype=np.int64)
    E = tbl.n_seg
    lo, hi = np.empty(E, np.int64), np.empty(E, np.int64)
    for e in range(E):
        a, b, _ = slice(int(tbl.seg_start[e]) - 1, int(tbl.seg_end[e])).indices(int(lens[tbl.seg_contig[e]]))
        lo[e], hi[e] = a, max(a, b)
    nuc, off = coracle.splice(contigs, tbl.rec_seg_off, tbl.seg_contig, lo, hi, tbl.seg_strand)
    aa, aa_off, aa_len = coracle.splice_translate(nuc, off)
    return nuc.tobytes(), aa[:aa_off[-1]].tobytes(), np.diff(off), aa_len


def _check_plans(g, tbl, want, tune):
    from magot_b200 import engine
    nuc, prot, nuc_len, aa_len = want
    for k1 in (0, 1):
        tune(b"k1", k1)
        for emit in (0, 1, 2):
            tune(b"emit", emit)
            text, (nl, al) = engine.run_table(g, tbl, want_lengths=True)
            assert text == nuc, (k1, emit)
            assert np.array_equal(nl, nuc_len) and np.array_equal(al, aa_len), (k1, emit)
            assert engine.run_table(g, tbl, protein=True)[0] == prot, (k1, emit)
            assert engine.run_table_both(g, tbl, async_prepare=bool(emit & 1)) == (nuc, prot), (k1, emit)
        a, bn, bp = engine.run_products(g, tbl, tbl)
        assert a == nuc and bn == nuc and bp == prot, k1
    tune(b"emit", 0)
    tune(b"k1", 0)


def test_mask_then_plans(mg, tune):
    """K1 + K2 + K3 (every emit variant and both K1 variants, fused and one-launch emits) on a soft- and then hard-masked
    genome against the C oracle on the model's bytes; the hard mask turns first codons into NNN, which changes trimX."""
    rng = np.random.default_rng(130)
    p = np.array([4, 4, 4, 4, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1], dtype=np.float64)
    contigs = _random_contigs(rng, lens=(5000, 257, 33, 20000, 8), p=p / p.sum())
    lens = [len(c) for c in contigs]
    model = gm.Genome(contigs)
    g = _genome(contigs)
    try:
        _mask(g, model, _intervals(rng, lens)[::4])
        tbl = _plan_table(rng, model.bytes_list(), [])
        _check_plans(g, tbl, _plan_want(tbl, model.bytes_list()), tune)
        hard = [iv for iv in _intervals(rng, lens)[::5] if iv[2] - iv[1] >= 3]
        tbl = _plan_table(rng, model.bytes_list(), hard)
        before = _plan_want(tbl, model.bytes_list())
        _mask(g, model, hard, hard=True)
        want = _plan_want(tbl, model.bytes_list())
        assert (want[3] != before[3]).sum() > 10           # first codons turned into NNN: one residue fewer after trimX
        _check_plans(g, tbl, want, tune)
    finally:
        g.close()


def _six_want(contigs, min_aa, code):
    recs, aa = [], []
    for ci, c in enumerate(contigs):
        a, rows = gref.sixframe(c, min_aa, gref.table64(code))
        recs += [(ci,) + tuple(r) for r in rows]
        aa.append(a)
    return recs, b"".join(aa)


def _six_got(result):
    recs, aa = result
    return [tuple(int(v) for v in r) for r in recs[["contig", "frame", "minus", "start", "len"]].tolist()], aa


def _orf_got(result):
    recs, aa = result
    rows = [tuple(int(v) for v in r) for r in recs[["contig", "minus", "phase", "flags", "start_codon", "lo", "hi", "len",
                                                     "aa_off"]].tolist()]
    return rows, aa


ORF_ARGS = ((100, 1, ("ATG",), False), (30, 11, ("ATG", "GTG", "TTG"), True), (0, 6, ("ATG",), True))


def _k4_results(g, n, tune):
    from magot_b200 import orfs
    out = {}
    for code in (1, 6):
        for min_aa in (0, 100):
            for mode in ((2, 1, 0) if min_aa else (2,)):
                tune(b"six", mode)
                out[("six", code, min_aa, mode)] = _six_got(orfs.sixframe(g, 0, n, min_aa, genetic_code=code))
    tune(b"six", 2)
    for args in ORF_ARGS:
        out[("orf",) + args] = _orf_got(orfs.call_orfs(g, list(range(n)), args[0], args[1], args[2], args[3]))
    return out


def _k4_check(got, contigs):
    ids = list(range(len(contigs)))
    for key, value in got.items():
        if key[0] == "six":
            assert value == _six_want(contigs, key[2], key[1]), key
        else:
            min_aa, code, starts, partial = key[1:]
            assert value == orfcall_ref.call_list(contigs, ids, min_aa, code, starts, partial), key


def test_mask_then_orfs(mg, tune):
    """The six-frame scan (codes 1 and 6, every scan variant; both stop-codon indexes built before the mask) and ORF
    calling on a masked genome against gencode_ref / orfcall_ref on the model's bytes.  A soft mask changes no result:
    K4 ignores case, and R/Y/K/M (listed as exceptions once lower-cased) are never part of a start or stop codon."""
    rng = np.random.default_rng(140)
    alpha = np.frombuffer(b"ACGTACGTACGTACGTacgtNRYKMrW", dtype=np.uint8)
    contigs = _random_contigs(rng, lens=(60000, 33, 9001, 257, 0, 30000), alpha=alpha)
    lens = [len(c) for c in contigs]
    n = len(contigs)
    model = gm.Genome(contigs)
    g = _genome(contigs)
    try:
        base = _k4_results(g, n, tune)                      # builds the table-1 and the table-6 stop-codon index
        _k4_check(base, model.bytes_list())
        _mask(g, model, _intervals(rng, lens), upper_first=True)
        _mask(g, model, _intervals(rng, lens)[::2])
        assert _k4_results(g, n, tune) == base
        _mask(g, model, _intervals(rng, lens)[::6], hard=True)
        got = _k4_results(g, n, tune)
        assert got != base
        _k4_check(got, model.bytes_list())
    finally:
        g.close()


def test_emit_device_matches_host(mg):
    """mg_orfcall_emit_device / mg_sixframe_emit_device into torch buffers equal mg_orfcall_emit / mg_sixframe_emit,
    records and residues, on a masked genome."""
    import torch
    from magot_b200 import _lib, orfs
    lib = _lib.lib
    rng = np.random.default_rng(150)
    alpha = np.frombuffer(b"ACGTACGTacgtNRY", dtype=np.uint8)
    contigs = _random_contigs(rng, lens=(80000, 5000, 31), alpha=alpha)
    model = gm.Genome(contigs)
    g = _genome(contigs)
    ids = np.arange(3, dtype=np.int64)
    try:
        _mask(g, model, _intervals(rng, [len(c) for c in contigs])[::3], hard=True)
        for kind in ("orf", "six"):
            n_orf, n_bytes = ctypes.c_int64(0), ctypes.c_int64(0)
            if kind == "orf":
                _lib.check(lib.mg_orfcall_count(g.handle, 3, ctypes.c_void_p(ids.ctypes.data), 20, None, None, 1,
                                                ctypes.byref(n_orf), ctypes.byref(n_bytes), None))
                dtype, emit, emit_dev = orfs.ORFCALL_DTYPE, lib.mg_orfcall_emit, lib.mg_orfcall_emit_device
            else:
                _lib.check(lib.mg_sixframe_count(g.handle, 0, 3, 20, ctypes.byref(n_orf), ctypes.byref(n_bytes), None))
                dtype, emit, emit_dev = orfs.ORF_DTYPE, lib.mg_sixframe_emit, lib.mg_sixframe_emit_device
            R, B = n_orf.value, n_bytes.value
            assert R > 100
            recs = np.zeros(R, dtype=dtype)
            aa = np.empty(B, dtype=np.uint8)
            _lib.check(emit(g.handle, ctypes.c_void_p(aa.ctypes.data), ctypes.c_void_p(recs.ctypes.data), None))
            d_aa = torch.full(((B + 15) // 16 * 16,), 255, dtype=torch.uint8, device="cuda")
            d_recs = torch.zeros(R * dtype.itemsize, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            _lib.check(emit_dev(g.handle, ctypes.c_void_p(d_aa.data_ptr()), ctypes.c_void_p(d_recs.data_ptr()), None))
            _lib.check(lib.mg_stream_sync(0, None))
            assert d_aa[:B].cpu().numpy().tobytes() == aa.tobytes(), kind
            assert d_recs.cpu().numpy().tobytes() == recs.tobytes(), kind
        want = orfcall_ref.call_list(model.bytes_list(), [0, 1, 2], 20, 1, ("ATG",), True)
        assert _orf_got(orfs.call_orfs(g, [0, 1, 2], 20, partial=True)) == want
    finally:
        g.close()


# ---- 5: K6 AT flags -------------------------------------------------------------------------------------------------------

def _at_flags(g, ci, lo, hi):
    from magot_b200 import _lib
    out = np.full(max(hi - lo, 1), 7, dtype=np.uint8)
    _lib.check(_lib.lib.mg_genome_at_flags(g.handle, ci, lo, hi, ctypes.c_void_p(out.ctypes.data), None))
    return out[:hi - lo]


def test_at_flags_random(mg):
    """Any lo that is a multiple of 8 and any hi (the partial last word included), on exception and IUPAC bytes, before and
    after a soft and a hard mask."""
    rng = np.random.default_rng(160)
    contigs = _random_contigs(rng) + _random_contigs(rng, lens=rng.integers(0, 5000, size=6))
    lens = [len(c) for c in contigs]
    model = gm.Genome(contigs)
    g = _genome(contigs)
    try:
        for step in range(3):
            if step == 1:
                _mask(g, model, _intervals(rng, lens)[::2], upper_first=True)
            if step == 2:
                _mask(g, model, _intervals(rng, lens)[::3], hard=True)
            for ci, L in enumerate(lens):
                ranges = [(0, L), (L // 8 * 8, L)]
                for _ in range(12):
                    lo = 8 * int(rng.integers(0, L // 8 + 1))
                    ranges.append((lo, int(rng.integers(lo, L + 1))))
                for lo, hi in ranges:
                    assert np.array_equal(_at_flags(g, ci, lo, hi), model.at_flags(ci, lo, hi)), (step, ci, lo, hi)
    finally:
        g.close()


def test_at_flags_past_staging_buffer(mg):
    """A contig a little longer than 2^28 bases: ranges longer than the 256 MiB staging buffer take two trips."""
    import torch
    from magot_b200 import engine, synth
    L = (1 << 28) + 4099
    dev = torch.device("cuda", 0)
    a = synth.synth_contig_device(L, 77, dev)
    g = engine.DeviceGenome([L], device=0)
    try:
        g.pack_device(0, a.data_ptr(), L)
        torch.cuda.synchronize()
        del a
        torch.cuda.empty_cache()
        g.finalize()
        seq = g.fetch(0, 0, L)
        want = gm.at_flags(seq)
        assert 0 < int(want.sum()) < L
        for lo in (0, 4096):
            assert np.array_equal(_at_flags(g, 0, lo, L), want[lo:]), lo
        lo = (1 << 28) - 64
        assert np.array_equal(_at_flags(g, 0, lo, L - 3), want[lo:L - 3])
    finally:
        g.close()


# ---- 6: argument checks --------------------------------------------------------------------------------------------------

def _snapshot(g, lens):
    return [(g.fetch(ci, 0, L), g.fetch(ci, 0, L, True)) for ci, L in enumerate(lens)]


def test_mask_argument_checks(mg):
    """Every rejected call raises MagotError and leaves the genome unchanged, and a count made before it stays valid."""
    from magot_b200 import _lib, engine
    from magot_b200._lib import MagotError
    lib = _lib.lib
    rng = np.random.default_rng(170)
    contigs = _random_contigs(rng, lens=(100, 64, 9))
    lens = [len(c) for c in contigs]
    g = _genome(contigs)
    try:
        snap = _snapshot(g, lens)
        n_exc = g.finalize()
        n_orf, n_bytes = ctypes.c_int64(0), ctypes.c_int64(0)
        _lib.check(lib.mg_sixframe_count(g.handle, 0, 3, 0, ctypes.byref(n_orf), ctypes.byref(n_bytes), None))
        bad = [(3, 0, 1), (-1, 0, 1), (0, 5, 4), (1, 0, 65), (2, 9, 10), (0, -1, 3)]
        for iv in bad:
            for hard in (False, True):
                for upper_first in (False, True):
                    with pytest.raises(MagotError):
                        g.mask(*_cols([(0, 0, 50), iv]), hard=hard, upper_first=upper_first)
                    assert _snapshot(g, lens) == snap, (iv, hard, upper_first)
        aa = np.empty(max(n_bytes.value, 1), dtype=np.uint8)
        _lib.check(lib.mg_sixframe_emit(g.handle, ctypes.c_void_p(aa.ctypes.data), None, None))
        assert g.finalize() == n_exc
        for ci, lo, hi in ((0, 3, 50), (0, 1, 8), (3, 0, 8), (-1, 0, 8), (0, 16, 8), (1, 0, 65), (2, 8, 10)):
            with pytest.raises(MagotError):
                _at_flags(g, ci, lo, hi)
        assert _snapshot(g, lens) == snap
        # before finalize: a mask and AT flags are refused; finalize then gives the packed bytes
        h = engine.DeviceGenome(lens, device=0)
        try:
            for i, c in enumerate(contigs):
                h.pack(i, np.frombuffer(c, dtype=np.uint8))
            with pytest.raises(MagotError):
                h.mask([0], [0], [50])
            with pytest.raises(MagotError):
                _at_flags(h, 0, 0, 8)
            h.finalize()
            assert _snapshot(h, lens) == snap
        finally:
            h.close()
    finally:
        g.close()


# ---- 7: emits after a genome change --------------------------------------------------------------------------------------

def _change(g, model, rng, how):
    lens = [len(c) for c in model.contigs]
    if how == "mask":
        _mask(g, model, [(0, 0, lens[0] // 2), (1, 3, lens[1])], hard=True)
    elif how == "soft":
        _mask(g, model, [(0, 0, lens[0] // 2)])
    elif how in ("pack", "repack"):
        new = _random_contigs(rng, lens=(lens[1],), alpha=np.frombuffer(b"ACGTN", dtype=np.uint8))[0]
        g.pack(1, np.frombuffer(new, dtype=np.uint8))
        model.contigs[1][:] = new
        model.listed[1][:] = False
        if how == "repack":
            g.finalize()


@pytest.mark.parametrize("how", ["mask", "soft", "pack", "repack"])
def test_stale_count_emits(mg, how):
    """A six-frame or ORF-call count, then a pack / finalize / mask, then an emit: MG_ESTATE from the host and the device
    emits; a new count gives the model's result."""
    import torch
    from magot_b200 import _lib, orfs
    lib = _lib.lib
    rng = np.random.default_rng(180)
    contigs = _random_contigs(rng, lens=(30000, 20000), alpha=np.frombuffer(b"ACGTACGTacgtN", dtype=np.uint8))
    model = gm.Genome(contigs)
    g = _genome(contigs)
    ids = np.arange(2, dtype=np.int64)
    d_buf = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    h_aa = np.empty(1 << 20, dtype=np.uint8)
    h_recs = np.zeros(1 << 14, dtype=orfs.ORFCALL_DTYPE)
    try:
        for kind in ("six", "orf"):
            n_orf, n_bytes = ctypes.c_int64(0), ctypes.c_int64(0)
            if kind == "six":
                _lib.check(lib.mg_sixframe_count(g.handle, 0, 2, 30, ctypes.byref(n_orf), ctypes.byref(n_bytes), None))
                emits = (lib.mg_sixframe_emit, lib.mg_sixframe_emit_device)
            else:
                _lib.check(lib.mg_orfcall_count(g.handle, 2, ctypes.c_void_p(ids.ctypes.data), 30, None, None, 1,
                                                ctypes.byref(n_orf), ctypes.byref(n_bytes), None))
                emits = (lib.mg_orfcall_emit, lib.mg_orfcall_emit_device)
            assert 0 < n_bytes.value < h_aa.size and 0 < n_orf.value < h_recs.size
            _change(g, model, rng, how)
            host = (ctypes.c_void_p(h_aa.ctypes.data), ctypes.c_void_p(h_recs.ctypes.data))
            dev = (ctypes.c_void_p(d_buf.data_ptr()), ctypes.c_void_p(d_buf.data_ptr() + (1 << 19)))
            for emit, bufs in zip(emits, (host, dev)):
                for args in (bufs, (bufs[0], None), (None, bufs[1])):
                    assert emit(g.handle, args[0], args[1], None) == MG_ESTATE, (kind, how)
                    assert "genome changed" in _lib.last_error()
            if how == "pack":
                g.finalize()
        assert _six_got(orfs.sixframe(g, 0, 2, 30)) == _six_want(model.bytes_list(), 30, 1)
        assert _orf_got(orfs.call_orfs(g, [0, 1], 30, partial=True)) == \
            orfcall_ref.call_list(model.bytes_list(), [0, 1], 30, 1, ("ATG",), True)
    finally:
        g.close()


def _plan_calls(lib, p, q, d, h):
    """Every call that reads a prepared plan `p` (q: a second, freshly prepared plan of the same genome)."""
    n = ctypes.c_int64(0)
    lens = np.empty(4096, dtype=np.int64)
    L = ctypes.c_void_p(lens.ctypes.data)
    return {
        "nuc_device": lambda: lib.mg_emit_nuc_device(p, d[0], None),
        "prot_device": lambda: lib.mg_emit_prot_device(p, d[1], None),
        "nuc_prot_device": lambda: lib.mg_emit_nuc_prot_device(p, d[0], d[1], None),
        "nuc_host": lambda: lib.mg_emit_nuc_host(p, h[0], None),
        "prot_host": lambda: lib.mg_emit_prot_host(p, h[1], None),
        "nuc_prot_host": lambda: lib.mg_emit_nuc_prot_host(p, h[0], h[1], None),
        "products_device_a": lambda: lib.mg_emit_products_device(p, d[0], q, d[2], d[3], None),
        "products_device_b": lambda: lib.mg_emit_products_device(q, d[0], p, d[2], d[3], None),
        "products_device_b_prot": lambda: lib.mg_emit_products_device(None, None, p, None, d[3], None),
        "products_host_a": lambda: lib.mg_emit_products_host(p, h[0], q, h[2], h[3], None),
        "products_host_b": lambda: lib.mg_emit_products_host(q, h[0], p, h[2], h[3], None),
        "totals": lambda: lib.mg_plan_totals(p, ctypes.byref(n), ctypes.byref(n), None),
        "lengths": lambda: lib.mg_plan_lengths(p, L, L, None),
    }


@pytest.mark.parametrize("prepare", ["prepare", "prepare_async", "prepare_deferred"])
def test_stale_plan_emits(mg, tune, prepare):
    """A plan prepared, then a mask of its genome, then any emit / totals / lengths: MG_ESTATE (the record pass fixed trimX
    skips and protein offsets from first codons the mask has turned into NNN).  Prepared again, it gives the model's text."""
    import torch
    from magot_b200 import _lib, engine
    lib = _lib.lib
    rng = np.random.default_rng(190)
    contigs = _random_contigs(rng, lens=(6000, 3000), alpha=np.frombuffer(b"ACGTACGTacgtN", dtype=np.uint8))
    model = gm.Genome(contigs)
    g = _genome(contigs)
    hard = [(0, 8 * k + 1, 8 * k + 41) for k in range(0, 700, 37)] + [(1, 8 * k + 5, 8 * k + 20) for k in range(0, 360, 29)]
    tbl = _plan_table(rng, contigs, hard, n_rec=200)
    cap = 1 << 21
    d_buf = torch.zeros(4 * cap, dtype=torch.uint8, device="cuda")
    h_buf = np.empty(4 * cap, dtype=np.uint8)
    d = [ctypes.c_void_p(d_buf.data_ptr() + k * cap) for k in range(4)]
    h = [ctypes.c_void_p(h_buf.ctypes.data + k * cap) for k in range(4)]
    try:
        for k1 in (0, 1):
            tune(b"k1", k1)
            p, q = engine.Plan(g, tbl), engine.Plan(g, tbl)
            try:
                if prepare == "prepare":
                    p.prepare()
                else:
                    p.prepare_async(defer_records=prepare == "prepare_deferred")
                calls = _plan_calls(lib, p.handle, q.handle, d, h)
                _mask(g, model, hard[k1::2], hard=True)
                q.prepare()
                for name, call in calls.items():
                    assert call() == MG_ESTATE, (prepare, k1, name)
                    assert "genome changed" in _lib.last_error(), name
                if prepare == "prepare_deferred":
                    assert lib.mg_plan_prepare_prot_async(p.handle, None) == MG_ESTATE
                lib.mg_stream_sync(0, None)
                nuc, prot, nuc_len, aa_len = _plan_want(tbl, model.bytes_list())
                p.prepare()
                assert p.emit_bytes() == nuc and p.emit_bytes(protein=True) == prot, (prepare, k1)
                nl, al = p.lengths()
                assert np.array_equal(nl, nuc_len) and np.array_equal(al, aa_len)
                assert calls["products_host_a"]() == 0 and calls["products_device_b"]() == 0
                lib.mg_stream_sync(0, None)
                if prepare != "prepare":
                    p.prepare_async(defer_records=prepare == "prepare_deferred")
                    if prepare == "prepare_deferred":
                        p.prepare_prot()
                    p.totals()
                    assert p.emit_bytes() == nuc and p.emit_bytes(protein=True) == prot, (prepare, k1, "again")
            finally:
                p.close()
                q.close()
    finally:
        g.close()


# ---- 8: mask_from_gff end to end ----------------------------------------------------------------------------------------

def _fasta_gff(rng):
    """Random FASTA (CRLF and LF lines, a repeated header, an empty record, headers with descriptions) and GFF text
    (CRLF lines, start = 0, negative, reversed and out-of-range coordinates, other feature types, lines with 5 and with
    more than 8 tabs, comments)."""
    alpha = np.frombuffer(b"ACGTACGTacgtNnRYKMrykmW*-", dtype=np.uint8)
    names = ["chr%d" % k for k in range(6)] + ["scaf_x", "u"]
    lens = {}
    fa = []
    for k, name in enumerate(names + ["chr2"]):                   # chr2 repeated: starts over
        L = 0 if name == "u" else int(rng.choice([1, 7, 31, 33, 250, 257, 1000, 4000]))
        lens[name] = L
        seq = alpha[rng.integers(0, alpha.size, size=L)].tobytes()
        eol = b"\r\n" if k % 2 else b"\n"
        fa.append((">%s%s" % (name, " some description" if k % 3 == 0 else "")).encode() + eol)
        w = int(rng.choice([10, 60, 61]))
        fa += [seq[i:i + w] + eol for i in range(0, L, w)]
    gff, clean = [], []
    for k in range(300):
        name = names[int(rng.integers(0, len(names)))]
        L = lens[name]
        kind = k % 7
        if kind == 0:
            a, b = 0, int(rng.integers(0, L + 3))
        elif kind == 1:
            a, b = int(rng.integers(-30, 0)), int(rng.integers(-10, L + 5))
        elif kind == 2:
            b = int(rng.integers(1, L + 2))
            a = b + int(rng.integers(1, 20))                     # reversed
        elif kind == 3:
            a = int(rng.integers(1, L + 10))
            b = a + int(rng.integers(0, 50))                     # may run past the end
        else:
            a = int(rng.integers(1, L + 1)) if L else 1
            b = min(L, a + int(rng.integers(0, 300)))
        feat = ["CDS", "CDS", "CDS", "exon", "gene"][int(rng.integers(0, 5))]
        cols = [name, "src", feat, str(a), str(b), ".", "+-"[k % 2], ".", "ID=f%d" % k]
        if k % 11 == 0:
            cols.append("extra")
        line = "\t".join(cols) + ("\r" if k % 4 == 0 else "")
        gff.append(line)
        if kind >= 4 or kind == 2:
            clean.append(line)
    gff += ["##gff-version 3", "chr1\tsrc\tCDS\t1\t5\t.", "# chr1\tsrc\tCDS\t1\t10"]
    rng.shuffle(gff)
    return b"".join(fa), "\n".join(gff) + "\n", "\n".join(clean + ["chr0\tsrc\tCDS\t1\t1\t.\t+\t.\t"]) + "\n"


def test_mask_from_gff_end_to_end(mg, tmp_path):
    import contextlib
    import io
    from magot_b200 import genome_tools as gt

    def run(*a, **k):
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            gt.mask_from_gff(*a, **k)
        return buf.getvalue().encode("latin-1")

    for seed in range(3):
        rng = np.random.default_rng(200 + seed)
        fa_text, gff_text, clean_text = _fasta_gff(rng)
        fa, gff, clean = tmp_path / "g.fa", tmp_path / "a.gff", tmp_path / "b.gff"
        fa.write_bytes(fa_text)
        gff.write_bytes(gff_text.encode())
        clean.write_bytes(clean_text.encode())
        for upper in ("True", "False"):
            for feat in ("CDS", "exon"):
                want = gm.mask_from_gff(fa_text, gff_text, "soft", upper, feat)
                assert run(str(fa), str(gff), overwrite_softmask=upper, feature_type=feat) == want, (seed, upper, feat)
                want = gm.mask_from_gff(fa_text, clean_text, "hard", upper, feat)
                assert run(str(fa), str(clean), mask_type="hard", overwrite_softmask=upper, feature_type=feat) == want
            with pytest.raises(NotImplementedError):
                gm.mask_from_gff(fa_text, gff_text, "hard", upper)
            with pytest.raises(NotImplementedError):
                run(str(fa), str(gff), mask_type="hard", overwrite_softmask=upper)
