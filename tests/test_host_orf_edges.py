"""The planted-ORF cases of tests/orf_plant.py against the references, without a GPU and without magot_b200: the builder's
intent against cdspredict_ref (candidates and the chosen ORF, at the prediction scan's lane and step edges, ties, partial ties,
min_aa at the winner), orfcall_ref (first starts at the ORF caller's step edges, stretches of 512k codons, stops on every
phase's last codon, the true-phase offsets the six-frame scan never flags) and cdscheck_ref (in-frame stops at 32 KB text tile
edges); the spliced payloads of '+' and '-' splits; and the references against each other: the longest ORF call of a strand is
the prediction of the whole contig on that strand, and every ORF call and every complete prediction passes the check."""
import numpy as np
import pytest

import cdscheck_ref as cref
import cdspredict_ref as pref
import orf_plant as op
import orfcall_ref as oref

CODES = (1, 2, 6, 11, 23)
START_SETS = (("ATG",), ("ATG", "GTG", "TTG"), op.SENSE)
PARTIALS = ((False, False), (True, False), (False, True), (True, True))
BAD = cref.NO_START | cref.NO_STOP | cref.INTERNAL_STOP | cref.PARTIAL_CODON


@pytest.mark.parametrize("code", CODES)
def test_predict_intent(code):
    rng = np.random.default_rng(100 + code)
    for which in START_SETS:
        stop, start = pref.code_sets(code, op.start_set(code, which))
        for name, s, cuts in op.predict_payloads(code, which, rng):
            s.verify()
            S = s.seq()
            for p5, p3 in PARTIALS:
                want = pref.candidates(S, stop, start, p5, p3)
                got = s.intent(False, p5, p3)
                assert sorted(got) == sorted(want), (name, which, p5, p3)
                for m in (1, op.W_MIN, op.W_MIN + 1):
                    assert op.winner(got, m) == pref.select(want, m), (name, which, p5, p3, m)
            for minus in (False, True):                  # the split record's payload is the planned one
                c, sg = op.split(S, cuts, minus, rng, 0)
                assert cref.payload([c], op.table([sg]), 0) == S


def test_predict_intent_names_the_edges():
    """The cases reach what they are named for: a winner at W_MIN, ties, and ORFs of 1 to 10 prediction steps."""
    rng = np.random.default_rng(7)
    cases = {name: s for name, s, _ in op.predict_payloads(1, ("ATG",), rng)}
    win = lambda n, p5=False, p3=False: op.winner(cases[n].intent(False, p5, p3), 1)      # noqa: E731
    assert win("min_aa0")[0] == op.W_MIN and win("tie-5partial")[1] == 40 and win("tie-5partial", True)[1] == 0
    t3 = cases["tie-3partial"].intent(False, False, True)
    assert win("tie-3partial", False, True)[1] == 40 and sorted(c[0] for c in t3 if not c[3])[-1] == op.W_MIN
    for name, lo in (("tie2-lane", 100), ("tie3-lanes", 100), ("tie2-steps", 30), ("tie3-steps", 119)):
        w = win(name)
        assert w[1] == lo and sum(1 for c in cases[name].intent() if c[0] == w[0]) >= 2
    for k in (1, 2, 3, 10):
        n_aa, lo, hi, _ = win("steps%d" % k)
        assert (k - 1) * op.PRD_STEP < hi - lo <= k * op.PRD_STEP


def _calls_ref(contigs, ids, min_aa, code, starts, partial):
    recs, _ = oref.call_list(contigs, ids, min_aa, code, starts, partial)
    return recs


@pytest.mark.parametrize("code", CODES)
def test_call_intent(code):
    rng = np.random.default_rng(200 + code)
    for which in START_SETS:
        starts = op.start_set(code, which)
        for name, s in op.call_contigs(code, which, rng):
            s.verify()
            for partial in (False, True):
                for m in (0, 1, 100):
                    recs = _calls_ref([s.seq()], [0], m, code, starts, partial)
                    got = sorted((r[1], r[2], r[5], r[6], r[7], r[3] == 0) for r in recs)
                    assert got == op.calls(s, m, partial), (name, which, partial, m)


def test_phase1_first_codon_stop():
    """DESIGN section 4: the codon at plus offset 1 and at minus offset L - 4 is a stop here; the ORFs after it are the same
    whether or not it counts, since the stretch it would open has no start before the planted one."""
    rng = np.random.default_rng(3)
    for code in CODES:
        for name, s in op.call_contigs(code, ("ATG",), rng):
            if not name.startswith("phase1"):
                continue
            S = s.seq()
            plus = oref.stream_orfs(S, 0, 1, 0, code, ("ATG",), True)
            minus = oref.stream_orfs(S, 1, 1, 0, code, ("ATG",), True)
            assert [(o[2], o[4]) for o in plus] == [(16, 120)]
            assert [(o[4], o[0]) for o in minus] == [((s.n - 1) // 3 - 9, 1)]


@pytest.mark.parametrize("framing", [False, True])
def test_check_intent(framing):
    rng = np.random.default_rng(5)
    for code in CODES:
        recs = op.check_records(code, rng, framing)
        contigs, segs = [], []
        for s, cuts, _ in recs:
            s.verify()
            c, sg = op.split(s.seq(), cuts, len(segs) % 3 == 2, rng, len(contigs))
            contigs.append(c)
            segs.append(sg)
        got, _, _ = cref.check(contigs, op.table(segs), code, ("ATG",))
        for (s, _, stops), g in zip(recs, got):
            assert g["n_stop"] == len(stops) + 1 and g["first_stop"] == min(stops + [s.n // 3 - 1])
            assert g["flags"] & ~cref.NONCANONICAL_SPLICE == (cref.INTERNAL_STOP if stops else 0) and g["start_codon"] == 14 and g["rem"] == 0


def _cross_genome(code, which, rng):
    contigs = [s.seq(rng if k % 2 else None) for k, (_, s) in enumerate(op.call_contigs(code, which, rng))]
    return contigs + op.random_contigs(rng)


def _longest_per_strand(recs, L, c, minus):
    mine = [(r[7], -(L - r[6] if minus else r[5]), r) for r in recs if r[0] == c and r[1] == minus]
    return max(mine)[2] if mine else None


@pytest.mark.parametrize("code", CODES)
def test_references_agree(code):
    """orfcall_ref against cdspredict_ref (whole contigs) and cdscheck_ref (every call as a record)."""
    rng = np.random.default_rng(300 + code)
    for which in START_SETS:
        starts = op.start_set(code, which)
        contigs = _cross_genome(code, which, rng)
        ids = list(range(len(contigs)))
        whole = op.table([[(c, 1, len(contigs[c]), m)] for c in ids for m in (0, 1)])
        for partial in (False, True):
            for m in (1, 30):
                recs = _calls_ref(contigs, ids, m, code, starts, partial)
                pr, ps = pref.predict(contigs, whole, code, starts, m, False, partial)
                for k in range(whole.n_rec):
                    c, minus = k // 2, k % 2
                    best = _longest_per_strand(recs, len(contigs[c]), c, minus)
                    if best is None:
                        assert pr[k]["n_aa"] == 0
                        continue
                    assert (pr[k]["n_aa"], pr[k]["start_codon"], ps[k][:2]) == (best[7], best[4], (best[5], best[6]))
            tbl = op.table([[(r[0], r[5] + 1, r[6], r[1])] for r in recs])
            chk, _, _ = cref.check(contigs, tbl, code, starts)
            for r, g in zip(recs, chk):
                if r[3] == 0:
                    assert g["start_codon"] == r[4] and g["n_stop"] == 1 and g["first_stop"] == r[7] and g["rem"] == 0
                    assert g["flags"] & BAD == 0
                else:
                    assert g["flags"] & cref.NO_STOP and not g["flags"] & cref.INTERNAL_STOP


def test_complete_predictions_pass_the_check():
    """Every complete prediction of the planted multi-segment records, written back as CDS segments, checks clean."""
    rng = np.random.default_rng(11)
    for code in CODES:
        for which in START_SETS:
            starts = op.start_set(code, which)
            contigs, segs, _ = op.predict_genome(code, which, rng)
            tbl = op.table(segs)
            pr, ps = pref.predict(contigs, tbl, code, starts, 1, False, False)
            cds, n = [], 0
            for r in range(tbl.n_rec):
                if pr[r]["n_aa"] and pr[r]["type"] == 0:
                    e0, e1 = tbl.rec_seg_off[r], tbl.rec_seg_off[r + 1]
                    cds.append([(int(tbl.seg_contig[e]), ps[e][0] + 1, ps[e][1], int(tbl.seg_strand[e]))
                                for e in range(e0, e1) if ps[e][0] >= 0])
                    n += len(cds[-1]) > 1
            assert n > 20
            chk, _, _ = cref.check(contigs, op.table(cds), code, starts)
            for g in chk:
                assert g["flags"] & BAD == 0 and g["n_stop"] == 1 and g["first_stop"] == g["n_codons"] - 1
