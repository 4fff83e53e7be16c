"""The ORF finders on the device at their lane, step, window and tile edges, with ORFs planted by tests/orf_plant.py, against
the references and against each other.  CDS prediction (k_predict_scan: 16 positions a lane, PRD_STEP = 512 a warp step,
k_predict_map) against cdspredict_ref over five codes, three start sets, four partial combinations, min_aa at the winner, the
table and its antisense; ORF calling (k_orf_start: ORF_SPAN = 512 codons a step) against orfcall_ref under the three scan
variants; the six-frame scan (SIX_WIN = 96-base windows, SIX_BPT = 144 bases a thread, the fast path from SIX_FAST_MIN_AA = 48,
SIX_TILE = 73 728-base tiles) against coracle and gencode_ref; the check (CHK_SPAN = 48 positions a lane, MG_NUC_TILE = 32 KB
text tiles) against cdscheck_ref.  Then, with no reference: the prediction of a whole contig is its longest ORF call on that
strand, and every ORF call and every complete prediction of a spliced record passes the check."""
import numpy as np
import pytest

import cdscheck_ref as cref
import cdspredict_ref as pref
import coracle
import gencode_ref as gref
import orf_plant as op
import orfcall_ref as oref
from test_gpu_check import _genome, _table

pytestmark = pytest.mark.gpu

CODES = (1, 2, 6, 11, 23)
START_SETS = (("ATG",), ("ATG", "GTG", "TTG"), op.SENSE)
PARTIALS = ((False, False), (True, False), (False, True), (True, True))
BAD = cref.NO_START | cref.NO_STOP | cref.INTERNAL_STOP | cref.PARTIAL_CODON
SIX_MIN_AA = (48, 96, 97, 128)


@pytest.fixture(scope="module")
def mg():
    import magot_b200
    return magot_b200


@pytest.fixture()
def six_mode(mg):
    from magot_b200 import _lib
    yield lambda v: _lib.check(_lib.lib.mg_tune(b"six", v))
    _lib.check(_lib.lib.mg_tune(b"six", 2))


def _plan(g, tbl, code):
    from magot_b200 import engine, gencode
    plan = engine.Plan(g, tbl)
    if code != 1:
        plan.set_codon_table(gencode.codon64(code))
    plan.prepare(trimx=False)
    return plan


@pytest.mark.parametrize("code", CODES)
def test_predict_edges(mg, code):
    from magot_b200 import gencode, genome
    rng = np.random.default_rng(400 + code)
    for which in START_SETS:
        starts = op.start_set(code, which)
        contigs, segs, _ = op.predict_genome(code, which, rng)
        tbl = _table(segs, framing=False)
        g = _genome(contigs)
        try:
            for t in (tbl, genome.antisense_table(tbl)):
                plan = _plan(g, t, code)
                cache = {}
                for p5, p3 in PARTIALS:
                    for m in (1, op.W_MIN, op.W_MIN + 1):
                        want = pref.predict(contigs, t, code, starts, m, p5, p3, cache)
                        msg = pref.compare(*plan.predict_cds(m, gencode.start64(starts, code), p5, p3), *want)
                        assert msg is None, (which, p5, p3, m, msg)
                plan.close()
        finally:
            g.close()


def _rows(recs):
    return [tuple(int(v) for v in r) for r in recs[["contig", "minus", "phase", "flags", "start_codon", "lo", "hi", "len"]].tolist()]


def _call_genome(code, which, rng):
    return [s.seq(rng if k % 2 else None) for k, (_, s) in enumerate(op.call_contigs(code, which, rng))]


@pytest.mark.parametrize("code", CODES)
def test_orfcall_edges(mg, six_mode, code):
    from magot_b200 import orfs
    rng = np.random.default_rng(500 + code)
    for which in START_SETS:
        starts = op.start_set(code, which)
        contigs = _call_genome(code, which, rng)
        n = len(contigs)
        g = _genome(contigs)
        perm = list(rng.permutation(n)) + [0]
        try:
            for partial in (False, True):
                for m in (0, 1, 100):
                    want = [r[:8] for r in oref.call_list(contigs, range(n), m, code, starts, partial)[0]]
                    for mode in (2, 1, 0):
                        six_mode(mode)
                        assert _rows(orfs.call_orfs(g, list(range(n)), m, code, starts, partial)[0]) == want, (which, partial, m, mode)
                    six_mode(2)
                    want = [r[:8] for r in oref.call_list(contigs, perm, m, code, starts, partial)[0]]
                    assert _rows(orfs.call_orfs(g, perm, m, code, starts, partial)[0]) == want, (which, partial, m, "list")
        finally:
            g.close()


@pytest.mark.parametrize("code", (1, 2, 6))
def test_sixframe_edges(mg, six_mode, code):
    from magot_b200 import orfs
    rng = np.random.default_rng(600 + code)
    contigs = [s.seq(rng if k % 2 else None) for k, s in enumerate(op.six_contigs(code, rng, SIX_MIN_AA))]
    n = len(contigs)
    g = _genome(contigs)
    try:
        for m in (46, 47, 48, 49) + SIX_MIN_AA:
            per = []
            for c in contigs:
                if code == 1:
                    aa, r = coracle.sixframe(c, m)
                    per.append((aa, [tuple(int(v) for v in x) for x in r]))
                else:
                    per.append(gref.sixframe(c, m, gref.table64(code)))
            want_aa = b"".join(p[0] for p in per)
            want = [(c,) + tuple(x) for c in range(n) for x in per[c][1]]
            if m in SIX_MIN_AA:                           # the planted pairs reach min_aa exactly
                assert any(x[-1] == m for x in want) and any(x[-1] == m + 1 for x in want)
            for mode in (2, 1, 0):
                six_mode(mode)
                recs, aa = orfs.sixframe(g, 0, n, m, genetic_code=code)
                got = [(int(r["contig"]), int(r["frame"]), int(r["minus"]), int(r["start"]), int(r["len"])) for r in recs]
                assert aa == want_aa and got == want, (m, mode)
    finally:
        g.close()


@pytest.mark.parametrize("framing", [False, True])
def test_check_edges(mg, framing):
    from magot_b200 import gencode
    rng = np.random.default_rng(700 + framing)
    for code in (1, 2, 23):
        recs = op.check_records(code, rng, framing)
        contigs, segs = [], []
        for s, cuts, _ in recs:
            c, sg = op.split(s.seq(rng if len(segs) % 2 else None), cuts, len(segs) % 3 == 2, rng, len(contigs))
            contigs.append(c)
            segs.append(sg)
        tbl = _table(segs, framing=framing)
        g = _genome(contigs)
        try:
            plan = _plan(g, tbl, code)
            got = plan.check(gencode.start64(("ATG",), code), False, True, True)
            want = cref.check(contigs, tbl, code, ("ATG",))
            assert cref.compare(got[0], want[0]) is None, cref.compare(got[0], want[0])
            assert np.array_equal(got[1].astype(np.int64), want[1]) and np.array_equal(got[2], want[2])
            for (s, _, stops), r in zip(recs, got[0]):
                assert int(r["n_stop"]) == len(stops) + 1 and int(r["first_stop"]) == min(stops + [s.n // 3 - 1])
            plan.close()
        finally:
            g.close()


# ---- the finders against each other -------------------------------------------------------------------------------------

@pytest.mark.parametrize("code", CODES)
def test_predict_calls_and_check_agree(mg, code):
    from magot_b200 import gencode, orfs
    rng = np.random.default_rng(800 + code)
    for which in START_SETS:
        starts = op.start_set(code, which)
        s64 = gencode.start64(starts, code)
        contigs = _call_genome(code, which, rng) + op.random_contigs(rng)
        ids = list(range(len(contigs)))
        g = _genome(contigs)
        try:
            whole = _table([[(c, 1, len(contigs[c]), m)] for c in ids for m in (0, 1)], framing=False)
            plan = _plan(g, whole, code)
            for partial in (False, True):
                calls, _ = orfs.call_orfs(g, ids, 30, code, starts, partial)
                pr, ps = plan.predict_cds(30, s64, False, partial)
                for k in range(whole.n_rec):
                    c, minus = k // 2, k % 2
                    L = len(contigs[c])
                    mine = [(int(r["len"]), -(L - int(r["hi"]) if minus else int(r["lo"])), i)
                            for i, r in enumerate(calls) if r["contig"] == c and r["minus"] == minus]
                    if not mine:
                        assert int(pr["n_aa"][k]) == 0, (which, partial, k)
                        continue
                    b = calls[max(mine)[2]]
                    assert (int(pr["n_aa"][k]), int(pr["start_codon"][k]), int(ps["lo"][k]), int(ps["hi"][k])) == \
                        (int(b["len"]), int(b["start_codon"]) & 0xFF, int(b["lo"]), int(b["hi"])), (which, partial, k)
                # every call as a one-segment record under the same table
                tbl = _table([[(int(r["contig"]), int(r["lo"]) + 1, int(r["hi"]), int(r["minus"]))] for r in calls], framing=False)
                cp = _plan(g, tbl, code)
                chk = cp.check(s64)[0]
                cp.close()
                for r, x in zip(calls, chk):
                    if int(r["flags"]) & 1:
                        assert int(x["flags"]) & cref.NO_STOP and not int(x["flags"]) & cref.INTERNAL_STOP
                    else:
                        assert int(x["start_codon"]) == int(r["start_codon"]) & 0xFF and int(x["n_stop"]) == 1
                        assert int(x["first_stop"]) == int(r["len"]) and int(x["rem"]) == 0 and int(x["flags"]) & BAD == 0
            plan.close()
        finally:
            g.close()
        # every complete prediction of the planted spliced records, written back as CDS segments
        contigs, segs, _ = op.predict_genome(code, which, rng)
        tbl = _table(segs, framing=False)
        g = _genome(contigs)
        try:
            plan = _plan(g, tbl, code)
            pr, ps = plan.predict_cds(1, s64, False, False)
            plan.close()
            cds = []
            for r in range(tbl.n_rec):
                if int(pr["n_aa"][r]) and int(pr["type"][r]) == 0:
                    cds.append([(int(tbl.seg_contig[e]), int(ps["lo"][e]) + 1, int(ps["hi"][e]), int(tbl.seg_strand[e]))
                                for e in range(tbl.rec_seg_off[r], tbl.rec_seg_off[r + 1]) if int(ps["lo"][e]) >= 0])
            assert sum(len(x) > 1 for x in cds) > 20
            cp = _plan(g, _table(cds, framing=False), code)
            for x in cp.check(s64)[0]:
                assert int(x["flags"]) & BAD == 0 and int(x["n_stop"]) == 1 and int(x["first_stop"]) == int(x["n_codons"]) - 1
            cp.close()
        finally:
            g.close()
