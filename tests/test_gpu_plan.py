"""K1 (the plan passes) at the block boundaries of its tiling, against a Python model of the reference's slicing.

The piece pass works on blocks of BLOCK consecutive pieces and maps each piece to its record inside the block; the record pass
gives each thread several records.  These tables put long records, runs of empty records, clamped-away and negative
coordinates and literal pieces on both sides of block boundaries, and check the two texts, mg_plan_lengths and
mg_plan_totals, through mg_plan_prepare and mg_plan_prepare_async."""
import numpy as np
import pytest

import magot_oracle as mo

pytestmark = pytest.mark.gpu

BLOCK = 2048                      # pieces per block of the piece pass (PLAN_TILE in mg_plan.cu)
CONTIG_LENS = [7_001, 300, 12_345]


@pytest.fixture(scope="module")
def genome():
    from magot_b200 import engine
    rng = np.random.default_rng(5)
    contigs = [np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n)].copy() for n in CONTIG_LENS]
    contigs[0][100:110] = np.frombuffer(b"NNRYKMacgt", dtype=np.uint8)
    g = engine.DeviceGenome([a.size for a in contigs], device=0)
    for i, a in enumerate(contigs):
        g.pack(i, a)
    g.finalize()
    yield g, [a.tobytes().decode("latin-1") for a in contigs]
    g.close()


@pytest.fixture()
def tune():
    from magot_b200 import _lib

    def set_(key, v):
        _lib.check(_lib.lib.mg_tune(key.encode(), v))
    yield set_
    set_("emit", 0)
    set_("k1", 0)


def make_table(recs, rng):
    """RecordTable of `recs` (lists of (contig, start, end, minus)), each record framed by a literal prefix of 0..6 bytes and
    a suffix of 0..2 bytes."""
    from magot_b200 import engine
    rec_off, cid, st, en, sd = [0], [], [], [], []
    for r in recs:
        for (c, a, b, m) in r:
            cid.append(c); st.append(a); en.append(b); sd.append(m)
        rec_off.append(len(cid))
    R = len(recs)
    pre = rng.integers(0, 7, size=R).astype(np.int32)
    suf = rng.integers(0, 3, size=R).astype(np.int32)
    lit_off = np.concatenate([[0], np.cumsum(pre.astype(np.int64) + suf)])[:R].astype(np.int64)
    lit = rng.integers(65, 91, size=int(pre.sum() + suf.sum())).astype(np.uint8)
    return engine.RecordTable(rec_off, cid, st, en, sd, lit_off, pre, suf, lit)


def model(tbl, recs, texts):
    """Nucleotide text, protein text and per-record lengths as the reference computes them (Python slices, translate with
    the leading-X trim)."""
    nuc, prot, nl, al = [], [], [], []
    for i, r in enumerate(recs):
        s = "".join(mo.reverse_compliment(texts[c][a - 1:b]) if m else texts[c][a - 1:b] for (c, a, b, m) in r)
        t = mo.translate(s)
        p0, pre, suf = int(tbl.rec_lit_off[i]), int(tbl.rec_pre_len[i]), int(tbl.rec_suf_len[i])
        head = tbl.lit[p0:p0 + pre].tobytes().decode()
        tail = tbl.lit[p0 + pre:p0 + pre + suf].tobytes().decode()
        nuc.append(head + s + tail)
        prot.append(head + (t or "") + tail)
        nl.append(len(s))
        al.append(-1 if t is None else len(t))
    return "".join(nuc).encode("latin-1"), "".join(prot).encode("latin-1"), nl, al


def check(g, texts, recs, seed=0):
    import torch
    from magot_b200 import engine
    rng = np.random.default_rng(seed)
    tbl = make_table(recs, rng)
    want_n, want_p, want_nl, want_al = model(tbl, recs, texts)
    plan = engine.Plan(g, tbl)
    assert plan.prepare() == (len(want_n), len(want_p))
    nl, al = plan.lengths()
    assert list(nl) == want_nl and list(al) == want_al
    assert plan.emit_host(False).tobytes() == want_n
    assert plan.emit_host(True).tobytes() == want_p
    # the same plan again without the host round trip, deferred record pass; tight capacities (the host-side bound of
    # capacities() does not follow negative coordinates that wrap around a contig)
    cap_n, cap_p = len(want_n), len(want_p)
    plan.prepare_async(cap_n, cap_p, defer_records=True)
    out_n = torch.zeros((cap_n + 31) // 32 * 32 + 32, dtype=torch.uint8, device="cuda")
    out_p = torch.zeros((cap_p + 31) // 32 * 32 + 32, dtype=torch.uint8, device="cuda")
    plan.emit_device(out_n.data_ptr(), protein=False)
    assert plan.totals() == (len(want_n), 0)
    plan.prepare_prot()
    plan.emit_device(out_p.data_ptr(), protein=True)
    assert plan.totals() == (len(want_n), len(want_p))
    nl, al = plan.lengths()
    assert list(nl) == want_nl and list(al) == want_al
    assert out_n[:len(want_n)].cpu().numpy().tobytes() == want_n
    assert out_p[:len(want_p)].cpu().numpy().tobytes() == want_p
    plan.close()
    return tbl


def seg(rng, kind="plain"):
    """One segment: plain, clamped away (past the contig end, or start > end) or with negative coordinates."""
    c = int(rng.integers(0, len(CONTIG_LENS)))
    L = CONTIG_LENS[c]
    m = int(rng.integers(0, 2))
    if kind == "plain":
        a = int(rng.integers(1, L))
        return (c, a, min(L, a + int(rng.integers(0, 40))), m)
    if kind == "away":
        return [(c, L + 5, L + 50, m), (c, 30, 10, m), (c, L + 1, L + 1, m)][int(rng.integers(0, 3))]
    a = -int(rng.integers(1, 60))                     # negative: Python slice semantics count from the contig's end
    return [(c, a, -1, m), (c, a, int(rng.integers(1, 90)), m), (c, 5, a, m), (c, 0, 7, m)][int(rng.integers(0, 4))]


def random_recs(rng, n_rec, p_away=0.1, p_neg=0.1, max_seg=9):
    recs = []
    for _ in range(n_rec):
        n = int(rng.integers(0, max_seg + 1))
        kinds = rng.choice(["plain", "away", "neg"], size=n, p=[1 - p_away - p_neg, p_away, p_neg])
        recs.append([seg(rng, k) for k in kinds])
    return recs


def n_piece(recs):
    return sum(len(r) for r in recs) + 2 * len(recs)


def pad_to(recs, target, rng):
    """Append records so the table has exactly `target` pieces (one-segment records, then one of 0..2 segments)."""
    recs = list(recs)
    while target - n_piece(recs) > 4:
        recs.append([seg(rng)])
    rest = target - n_piece(recs)
    assert rest != 1, "start further below the target"
    if rest >= 2:
        recs.append([seg(rng) for _ in range(rest - 2)])
    assert n_piece(recs) == target
    return recs


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("delta", [-1, 0, 1])
def test_piece_count_around_block_multiples(genome, k, delta):
    g, texts = genome
    rng = np.random.default_rng(100 * k + delta)
    recs = pad_to(random_recs(rng, 200), k * BLOCK + delta, rng)
    check(g, texts, recs, seed=k)


def test_record_longer_than_blocks(genome):
    """One record of 9 000 segments (more than two blocks) between ordinary ones, and one that starts a block exactly."""
    g, texts = genome
    rng = np.random.default_rng(7)
    head = random_recs(rng, 50)
    head = pad_to(head, BLOCK, rng)                  # the long record's prefix is the first piece of block 1
    long_rec = [seg(rng, k) for k in rng.choice(["plain", "away", "neg"], size=9_000, p=[0.8, 0.1, 0.1])]
    recs = head + [long_rec] + random_recs(rng, 400) + [[seg(rng) for _ in range(5_000)]]
    check(g, texts, recs, seed=7)


def test_runs_of_empty_records(genome):
    """Runs of records without segments (or with only clamped-away ones) longer than a block's pieces."""
    g, texts = genome
    rng = np.random.default_rng(8)
    away = [[seg(rng, "away") for _ in range(int(rng.integers(1, 4)))] for _ in range(2_500)]
    recs = random_recs(rng, 100) + [[] for _ in range(2 * BLOCK + 17)] + random_recs(rng, 100) + away + random_recs(rng, 60)
    recs += [[] for _ in range(BLOCK // 2 + 1)]
    check(g, texts, recs, seed=8)


@pytest.mark.parametrize("shift", [0, 1, 2, 3, 4])
def test_literals_and_odd_segments_at_block_edges(genome, shift):
    """Records of one segment each (3 pieces), shifted so prefix, segment and suffix pieces each land on pieces BLOCK - 2 ..
    BLOCK + 2 and 2 BLOCK - 2 .. 2 BLOCK + 2; the segments near the edges are clamped away or negative."""
    g, texts = genome
    rng = np.random.default_rng(20 + shift)
    recs = [[seg(rng) for _ in range(shift)]]
    while n_piece(recs) < 3 * BLOCK:
        p = n_piece(recs) + 1                          # piece of the next record's segment
        near = min(abs(p - BLOCK), abs(p - 2 * BLOCK)) <= 6
        kind = ["away", "neg", "plain"][int(rng.integers(0, 3))] if near else "plain"
        recs.append([seg(rng, kind)])
    check(g, texts, recs, seed=20 + shift)


def test_random_tables_many_blocks(genome):
    g, texts = genome
    rng = np.random.default_rng(9)
    recs = random_recs(rng, 6_000, p_away=0.15, p_neg=0.15, max_seg=14)
    check(g, texts, recs, seed=9)


def test_one_kb_table_with_streaming_emit(genome, tune):
    """The 1 KB block table the piece pass fills for the streaming K2 variant (mg_tune emit=2)."""
    g, texts = genome
    tune("emit", 2)
    rng = np.random.default_rng(10)
    recs = pad_to(random_recs(rng, 900, max_seg=12), 4 * BLOCK + 1, rng)
    check(g, texts, recs, seed=10)


def test_alternating_streams_deferred_records_no_join(genome):
    """One plan prepared 20 times, its piece pass on two streams in turn and its deferred record pass on a third, with no join
    between steps: a record pass may still run when the next piece pass starts, and each pass owns its look-back words."""
    import ctypes
    import torch
    from magot_b200 import engine
    g, texts = genome
    rng = np.random.default_rng(11)
    recs = random_recs(rng, 8_000, max_seg=12)
    tbl = make_table(recs, rng)
    want_n, want_p, want_nl, want_al = model(tbl, recs, texts)
    s = [torch.cuda.Stream() for _ in range(3)]
    sp = [ctypes.c_void_p(x.cuda_stream) for x in s]
    plan = engine.Plan(g, tbl, stream=sp[0])
    cap_n, cap_p = len(want_n) + 1000, len(want_p) + 1000
    out_n = torch.zeros((cap_n + 31) // 32 * 32 + 32, dtype=torch.uint8, device="cuda")
    out_p = torch.zeros((cap_p + 31) // 32 * 32 + 32, dtype=torch.uint8, device="cuda")
    plan.prepare_async(cap_n, cap_p)                  # first prepare: allocations
    torch.cuda.synchronize()
    done = None
    for i in range(20):
        a = s[i % 2]
        if done is not None:
            a.wait_event(done)                        # the plan's piece passes follow each other; record passes are not waited for
        plan.stream = sp[i % 2]
        plan.prepare_async(cap_n, cap_p, defer_records=True)
        plan.emit_device(out_n.data_ptr(), protein=False)
        done = torch.cuda.Event()
        done.record(a)
        s[2].wait_event(done)
        plan.prepare_prot(sp[2])
        plan.stream = sp[2]
        plan.emit_device(out_p.data_ptr(), protein=True)
    torch.cuda.synchronize()
    assert plan.totals() == (len(want_n), len(want_p))
    nl, al = plan.lengths()
    assert list(nl) == want_nl and list(al) == want_al
    assert out_n[:len(want_n)].cpu().numpy().tobytes() == want_n
    assert out_p[:len(want_p)].cpu().numpy().tobytes() == want_p
    plan.close()
