"""The device-resident step of config 4 against the C oracle: mg_plan_prepare_async with caller capacities, the deferred record
pass on another stream, K2 / K3 / K23, the one-launch mg_emit_products_device, back-to-back steps with no join between them,
and CUDA-graph capture and replay.

Every output buffer is poisoned before a step or a replay.  Afterwards [0, total) must equal the oracle's text and every byte
from round_up(total, 32) on must still be poison; a buffer whose product was skipped must be untouched."""
import ctypes

import numpy as np
import pytest

import coracle
import gencode_ref as ref

pytestmark = pytest.mark.gpu

POISON = 0xA5
LAGS = [0, 1, 20_000, 1_000_000]
_LEAKED = []                      # plans a refused capture may have left in an unknown state: never used or destroyed again


def pad(n):
    return (n + 31) // 32 * 32 + 32


def round_up32(n):
    return (n + 31) // 32 * 32


# ---- workload: a small twin of config 4 --------------------------------------------------------------------------------

def oracle_texts(contigs, tbl, code=None):
    """(nucleotide text, protein text) of a framed table: coracle.splice + coracle.splice_translate (or gencode_ref.translate
    under NCBI table `code`), with each record's literal prefix and suffix around its payload."""
    n_rec = tbl.n_rec
    if n_rec == 0:
        return b"", b""
    lens = np.array([a.size for a in contigs])
    lo = np.clip(tbl.seg_start - 1, 0, lens[tbl.seg_contig])
    hi = np.clip(tbl.seg_end, 0, lens[tbl.seg_contig])
    nuc, off = coracle.splice([a.tobytes() for a in contigs], tbl.rec_seg_off, tbl.seg_contig, lo, hi, tbl.seg_strand)
    if code is None:
        aa, aa_off, _ = coracle.splice_translate(nuc, off)
        prot = [aa[aa_off[r]:aa_off[r + 1]].tobytes() for r in range(n_rec)]
    else:
        table = ref.table64(code)
        prot = [ref.translate(nuc[off[r]:off[r + 1]].tobytes(), table) or b"" for r in range(n_rec)]
    tn, tp = [], []
    for r in range(n_rec):
        p0, pre, suf = int(tbl.rec_lit_off[r]), int(tbl.rec_pre_len[r]), int(tbl.rec_suf_len[r])
        head, tail = tbl.lit[p0:p0 + pre].tobytes(), tbl.lit[p0 + pre:p0 + pre + suf].tobytes()
        tn.append(head + nuc[off[r]:off[r + 1]].tobytes() + tail)
        tp.append(head + prot[r] + tail)
    return b"".join(tn), b"".join(tp)


class Twin(object):
    """6 Mbp 'human' genome with out-of-alphabet bytes, 3000 transcripts, exon and CDS tables framed as in bench.py."""

    def __init__(self):
        import torch
        from magot_b200 import engine, synth
        layout = synth.contig_layout("human", 6_000_000, 4)
        self.contigs = synth.synth_genome_host(layout, 4, n_mean=300)
        rng = np.random.default_rng(11)
        for a in self.contigs[:6]:
            idx = rng.integers(0, a.size, size=80)
            a[idx] = np.frombuffer(b"RYKMSWBDHVrykm*", dtype=np.uint8)[rng.integers(0, 15, size=80)]
        self.ann = synth.synth_annotation(layout, 3000, 4)
        self.g = engine.DeviceGenome([a.size for a in self.contigs], device=0)
        for i, a in enumerate(self.contigs):
            self.g.pack(i, a)
        self.g.finalize()
        self.tables = {"cds": self.ann.table("cds"), "exon": self.ann.table("exon")}
        self.want = {k: oracle_texts(self.contigs, t) for k, t in self.tables.items()}
        self.streams = tuple(torch.cuda.Stream() for _ in range(3))

    def plan(self, k, table=None):
        from magot_b200 import engine
        return engine.Plan(self.g, self.tables[k] if table is None else table, stream=sp(self.streams[0]))


@pytest.fixture(scope="module")
def twin():
    t = Twin()
    yield t
    import torch
    torch.cuda.synchronize()
    t.g.close()


@pytest.fixture()
def tune():
    from magot_b200 import _lib

    def set_(key, v):
        _lib.check(_lib.lib.mg_tune(key.encode(), v))
    yield set_
    set_("emit", 0)
    set_("k1", 0)
    set_("multi_lag", 0)


def sp(stream):
    return ctypes.c_void_p(stream.cuda_stream) if stream is not None else None


def P(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def lib():
    from magot_b200 import _lib
    return _lib.lib


def chk(rc):
    from magot_b200 import _lib
    _lib.check(rc)


def new_buf(n, stream):
    import torch
    with torch.cuda.stream(stream):
        return torch.empty(pad(n), dtype=torch.uint8, device="cuda")


def poison(bufs, stream):
    import torch
    with torch.cuda.stream(stream):
        for b in bufs:
            b.fill_(POISON)
    torch.cuda.synchronize()


def check_text(buf, want, what):
    """[0, len(want)) == want and poison from round_up(len, 32) on; want None: the buffer was skipped and is all poison."""
    got = buf.cpu().numpy()
    if want is None:
        bad = np.flatnonzero(got != POISON)
        assert bad.size == 0, "%s: skipped buffer written at byte %d" % (what, bad[0])
        return
    n = len(want)
    if got[:n].tobytes() != want:
        first = int(np.flatnonzero(got[:n] != np.frombuffer(want, dtype=np.uint8))[0])
        raise AssertionError("%s: text differs from the oracle at byte %d of %d" % (what, first, n))
    bad = np.flatnonzero(got[round_up32(n):] != POISON)
    assert bad.size == 0, "%s: byte %d written past the text (%d bytes)" % (what, round_up32(n) + bad[0], n)


# ---- the step (bench.py's Workload.step, restated) -----------------------------------------------------------------------

class Step(object):
    """Exon and CDS plans of the twin, capacities from the host tables (Plan.capacities), and the step of every mode."""

    def __init__(self, twin, codon64=None):
        from magot_b200 import _lib
        self.t, self._lib = twin, _lib
        self.s, self.sb, self.sc = twin.streams
        self.plans = {k: twin.plan(k) for k in ("cds", "exon")}
        if codon64 is not None:
            self.plans["cds"].set_codon_table(codon64)
        self.caps = {k: p.capacities() for k, p in self.plans.items()}

    def buffers(self):
        return {"cds_n": new_buf(self.caps["cds"][0], self.s), "cds_p": new_buf(self.caps["cds"][1], self.s),
                "exon_n": new_buf(self.caps["exon"][0], self.s)}

    def prepare_on(self, k, s, defer=False):
        flags = self._lib.MG_PROT_TRIMX | (self._lib.MG_PROT_DEFER if defer else 0)
        chk(lib().mg_plan_prepare_async(self.plans[k].handle, flags, self.caps[k][0], self.caps[k][1], sp(s)))

    def step(self, mode, defer, out):
        import torch
        L, h = lib(), {k: p.handle for k, p in self.plans.items()}
        s, sb, sc = self.s, self.sb, self.sc
        if mode == "fused":
            self.prepare_on("cds", s)
            chk(L.mg_emit_nuc_prot_device(h["cds"], P(out["cds_n"]), P(out["cds_p"]), sp(s)))
            self.prepare_on("exon", sb)
            chk(L.mg_emit_nuc_device(h["exon"], P(out["exon_n"]), sp(sb)))
            return
        if mode == "multi":
            self.prepare_on("exon", sb)
            self.prepare_on("cds", s)
            s.wait_stream(sb)
            chk(L.mg_emit_products_device(h["exon"], P(out["exon_n"]), h["cds"], P(out["cds_n"]), P(out["cds_p"]), sp(s)))
            return
        self.prepare_on("cds", s, defer=defer)
        e1 = torch.cuda.Event()
        e1.record(s)
        chk(L.mg_emit_nuc_device(h["cds"], P(out["cds_n"]), sp(s)))
        sc.wait_event(e1)
        if defer:
            chk(L.mg_plan_prepare_prot_async(h["cds"], sp(sc)))
        chk(L.mg_emit_prot_device(h["cds"], P(out["cds_p"]), sp(sc)))
        self.prepare_on("exon", sb, defer=defer)
        chk(L.mg_emit_nuc_device(h["exon"], P(out["exon_n"]), sp(sb)))

    def join(self):
        self.s.wait_stream(self.sb)
        self.s.wait_stream(self.sc)

    def capture(self, mode, defer, out):
        """The step as one CUDA graph, forked and joined with mg_stream_wait_stream as Workload.capture does it.  With
        defer, the CDS record pass (mg_plan_prepare_prot_async) runs on the forked stream_c inside the graph."""
        L, h = lib(), {k: p.handle for k, p in self.plans.items()}
        s, sb, sc = sp(self.s), sp(self.sb), sp(self.sc)
        chk(L.mg_graph_begin(0, s))
        try:
            chk(L.mg_stream_wait_stream(0, sb, s))
            if mode == "multi":
                self.prepare_on("exon", self.sb)
                self.prepare_on("cds", self.s)
                chk(L.mg_stream_wait_stream(0, s, sb))
                chk(L.mg_emit_products_device(h["exon"], P(out["exon_n"]), h["cds"], P(out["cds_n"]), P(out["cds_p"]), s))
            elif mode == "fused":
                self.prepare_on("exon", self.sb)
                chk(L.mg_emit_nuc_device(h["exon"], P(out["exon_n"]), sb))
                self.prepare_on("cds", self.s)
                chk(L.mg_emit_nuc_prot_device(h["cds"], P(out["cds_n"]), P(out["cds_p"]), s))
                chk(L.mg_stream_wait_stream(0, s, sb))
            else:
                self.prepare_on("exon", self.sb, defer=defer)
                chk(L.mg_emit_nuc_device(h["exon"], P(out["exon_n"]), sb))
                self.prepare_on("cds", self.s, defer=defer)
                chk(L.mg_stream_wait_stream(0, sc, s))
                chk(L.mg_emit_nuc_device(h["cds"], P(out["cds_n"]), s))
                if defer:
                    chk(L.mg_plan_prepare_prot_async(h["cds"], sc))
                chk(L.mg_emit_prot_device(h["cds"], P(out["cds_p"]), sc))
                chk(L.mg_stream_wait_stream(0, s, sb))
                chk(L.mg_stream_wait_stream(0, s, sc))
        finally:
            g = ctypes.c_void_p()
            chk(L.mg_graph_end(0, s, ctypes.byref(g)))
        return g

    def check(self, out, exon_records, want_cds=None, what=""):
        """All three texts, then mg_plan_totals of both plans (exon_records: the exon plan's record pass ran)."""
        import torch
        torch.cuda.synchronize()
        wc = self.t.want["cds"] if want_cds is None else want_cds
        we = self.t.want["exon"]
        check_text(out["cds_n"], wc[0], what + " cds nucleotide")
        check_text(out["cds_p"], wc[1], what + " cds protein")
        check_text(out["exon_n"], we[0], what + " exon nucleotide")
        assert self.plans["cds"].totals() == (len(wc[0]), len(wc[1])), what
        assert self.plans["exon"].totals() == (len(we[0]), len(we[1]) if exon_records else 0), what

    def close(self):
        import torch
        torch.cuda.synchronize()
        for p in self.plans.values():
            p.close()


STEP_CASES = ([("streams3", d, k1, e, 0) for d in (False, True) for k1 in (0, 1) for e in (0, 1, 2)] +
              [("fused", False, k1, 0, 0) for k1 in (0, 1)] +
              [("multi", False, k1, 0, lag) for k1 in (0, 1) for lag in LAGS])


def _exon_records(defer, k1):
    """Whether the step runs the exon plan's record pass: the one-launch K1 always does, the piece-parallel one unless deferred."""
    return not defer or k1 == 1


@pytest.mark.parametrize("mode,defer,k1,emit,lag", STEP_CASES)
def test_eager_step(twin, tune, mode, defer, k1, emit, lag):
    """One step of every mode and K1 / K2 variant: the streaming K2 needs its 1 KB block table, so `emit` is set before the
    prepare."""
    tune("emit", emit)
    tune("k1", k1)
    tune("multi_lag", lag)
    st = Step(twin)
    out = st.buffers()
    for rep in range(2):                                  # the second step re-prepares plans that already hold their tables
        poison(out.values(), twin.streams[0])
        st.step(mode, defer, out)
        st.join()
        st.check(out, _exon_records(defer, k1), what="%s step %d" % (mode, rep))
    st.close()


@pytest.mark.parametrize("mode,defer,k1", [("streams3", d, k1) for d in (False, True) for k1 in (0, 1)] +
                         [("multi", False, k1) for k1 in (0, 1)])
def test_back_to_back_steps(twin, tune, mode, defer, k1):
    """Six steps with no join between them, as the timed loop of bench.py issues them, each into its own buffers.  The next
    step re-prepares both plans while the emits of the previous one may still run on the other streams: they re-create the
    same tables, so every buffer set must hold the full texts.  A pass does not prove the absence of a race."""
    tune("k1", k1)
    st = Step(twin)
    sets = [st.buffers() for _ in range(6)]
    st.step(mode, defer, sets[0])                         # tables grown once
    st.join()
    for out in sets:
        poison(out.values(), twin.streams[0])
    for out in sets:
        st.step(mode, defer, out)
    st.join()
    for i, out in enumerate(sets):
        st.check(out, _exon_records(defer, k1), what="%s step %d of 6" % (mode, i))
    st.close()


# ---- CUDA graphs ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode,defer", [("streams3", False), ("streams3", True), ("fused", False), ("multi", False)])
@pytest.mark.parametrize("k1", [0, 1])
def test_graph_replay(twin, tune, mode, defer, k1):
    tune("k1", k1)
    st = Step(twin)
    out = st.buffers()
    st.step(mode, defer, out)                             # eager warm-up: every buffer a capture needs exists now
    st.join()
    poison(out.values(), twin.streams[0])
    g = st.capture(mode, defer, out)
    try:
        for rep in range(3):
            poison(out.values(), twin.streams[0])
            chk(lib().mg_graph_launch(0, g, sp(st.s)))
            st.check(out, _exon_records(defer, k1), what="%s replay %d" % (mode, rep))
    finally:
        lib().mg_graph_destroy(g)
    st.close()


def test_graph_replay_genetic_code_2(twin):
    """A graph whose CDS plan translates with NCBI table 2 (set before the warm-up): the protein text follows the code."""
    from magot_b200 import gencode
    st = Step(twin, codon64=gencode.codon64(2))
    want_cds = oracle_texts(twin.contigs, twin.tables["cds"], code=2)
    assert want_cds[0] == twin.want["cds"][0] and want_cds[1] != twin.want["cds"][1]
    out = st.buffers()
    st.step("streams3", False, out)
    st.join()
    poison(out.values(), twin.streams[0])
    g = st.capture("streams3", False, out)
    try:
        for rep in range(3):
            poison(out.values(), twin.streams[0])
            chk(lib().mg_graph_launch(0, g, sp(st.s)))
            st.check(out, True, want_cds=want_cds, what="code 2 replay %d" % rep)
    finally:
        lib().mg_graph_destroy(g)
    st.close()


def _expect_refused(fn):
    from magot_b200 import _lib
    with pytest.raises(_lib.MagotError) as e:
        fn()
    msg = str(e.value)
    assert "error %d" % -4 in msg and "outside the capture" in msg, msg


def _leak(*plans):
    for p in plans:
        _LEAKED.append(p.handle)
        p.handle = ctypes.c_void_p()                      # Plan.close / __del__ leave it alone


@pytest.mark.parametrize("case", ["first_prepare", "larger_capacity", "larger_products_grid"])
def test_capture_refuses_buffer_growth(twin, case):
    """Inside a capture a grown plan buffer would be a graph allocation that nothing frees (a second launch of the graph fails,
    and the plan would point at memory that does not exist before the first launch).  Such a call must fail with MG_ESTATE
    before it queues anything; the capture still ends, and its graph is destroyed without being launched.  After an eager
    run of the same calls, the capture succeeds and replays correctly."""
    import torch
    from magot_b200 import _lib
    L, s, flags = lib(), twin.streams[0], _lib.MG_PROT_TRIMX
    want_c, want_e = twin.want["cds"], twin.want["exon"]
    pc, pe = twin.plan("cds"), twin.plan("exon")
    caps_c, caps_e = pc.capacities(), pe.capacities()
    cap_c = (caps_c[0] + (10 << 20), caps_c[1] + (10 << 20)) if case == "larger_capacity" else caps_c   # hundreds of tiles more
    out = {"cds_n": new_buf(cap_c[0], s), "cds_p": new_buf(cap_c[1], s), "exon_n": new_buf(caps_e[0], s)}

    def calls(pc, pe):
        """what each case captures"""
        if case == "larger_products_grid":
            chk(L.mg_plan_prepare_async(pe.handle, flags, caps_e[0], caps_e[1], sp(s)))
            chk(L.mg_plan_prepare_async(pc.handle, flags, cap_c[0], cap_c[1], sp(s)))
            chk(L.mg_emit_products_device(pe.handle, P(out["exon_n"]), pc.handle, P(out["cds_n"]), P(out["cds_p"]), sp(s)))
        else:
            chk(L.mg_plan_prepare_async(pc.handle, flags, cap_c[0], cap_c[1], sp(s)))
            chk(L.mg_emit_nuc_prot_device(pc.handle, P(out["cds_n"]), P(out["cds_p"]), sp(s)))

    # refused: (a) a never-prepared plan; (b) capacities above those of the eager prepare; (c) a products grid above the lead
    # plan's order buffer (its eager emit wrote the exon text alone)
    if case == "larger_capacity":
        chk(L.mg_plan_prepare_async(pc.handle, flags, caps_c[0], caps_c[1], sp(s)))
    if case == "larger_products_grid":
        chk(L.mg_plan_prepare_async(pe.handle, flags, caps_e[0], caps_e[1], sp(s)))
        chk(L.mg_plan_prepare_async(pc.handle, flags, caps_c[0], caps_c[1], sp(s)))
        chk(L.mg_emit_products_device(pe.handle, P(out["exon_n"]), pc.handle, None, None, sp(s)))
    torch.cuda.synchronize()
    g = ctypes.c_void_p()
    chk(L.mg_graph_begin(0, sp(s)))
    try:
        _expect_refused(lambda: calls(pc, pe))
    finally:
        chk(L.mg_graph_end(0, sp(s), ctypes.byref(g)))
        L.mg_graph_destroy(g)
        _leak(pc, pe)

    # the same capture after an eager run of the same calls succeeds and replays twice
    pc, pe = twin.plan("cds"), twin.plan("exon")
    calls(pc, pe)
    torch.cuda.synchronize()
    chk(L.mg_graph_begin(0, sp(s)))
    try:
        calls(pc, pe)
    finally:
        chk(L.mg_graph_end(0, sp(s), ctypes.byref(g)))
    try:
        for rep in range(2):
            poison(out.values(), s)
            chk(L.mg_graph_launch(0, g, sp(s)))
            torch.cuda.synchronize()
            check_text(out["cds_n"], want_c[0], "%s replay %d cds nucleotide" % (case, rep))
            check_text(out["cds_p"], want_c[1], "%s replay %d cds protein" % (case, rep))
            check_text(out["exon_n"], want_e[0] if case == "larger_products_grid" else None, "%s replay %d exon" % (case, rep))
            assert pc.totals() == (len(want_c[0]), len(want_c[1]))
    finally:
        L.mg_graph_destroy(g)
    pc.close()
    pe.close()


# ---- mg_emit_products_device: outputs x lag x plan pairs x prepares -----------------------------------------------------

def _extra_tables(twin):
    """1-tile table, a table with no record, and one whose records hold 1-2 bases (protein text: framing only)."""
    from magot_b200 import engine
    cds = twin.tables["cds"]
    small = cds.slice(0, 8)
    empty = engine.RecordTable(np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(0, np.int64),
                               np.zeros(0, np.int8), np.zeros(0, np.int64), np.zeros(0, np.int32), np.zeros(0, np.int32),
                               np.zeros(0, np.uint8))
    rng = np.random.default_rng(5)
    n = 400
    nseg = rng.integers(0, 3, size=n)
    off = np.concatenate(([0], np.cumsum(nseg)))
    E = int(off[-1])
    cid = rng.integers(0, len(twin.contigs), size=E).astype(np.int32)
    Ls = np.array([a.size for a in twin.contigs], dtype=np.int64)[cid]
    st = rng.integers(1, Ls - 4)
    en = st + rng.integers(0, 2, size=E)                 # one segment: 1 or 2 bases
    two = np.flatnonzero(nseg == 2)
    en[off[two]] = st[off[two]]                          # two segments: one base each
    en[off[two] + 1] = st[off[two] + 1]
    pre = rng.integers(1, 30, size=n).astype(np.int32)
    suf = np.ones(n, dtype=np.int32)
    lit = rng.integers(33, 127, size=int(pre.sum() + suf.sum()), dtype=np.uint8)
    lit_off = np.concatenate(([0], np.cumsum(pre.astype(np.int64) + suf)[:-1]))
    tiny = engine.RecordTable(off, cid, st, en, rng.integers(0, 2, size=E).astype(np.int8), lit_off, pre, suf, lit)
    return {"small": small, "empty": empty, "tiny": tiny}


@pytest.fixture(scope="module")
def products(twin):
    tables = dict(twin.tables)
    tables.update(_extra_tables(twin))
    want = {k: (twin.want[k] if k in twin.want else oracle_texts(twin.contigs, t)) for k, t in tables.items()}
    for r in range(tables["tiny"].n_rec):                 # every payload of the tiny table has at most 2 bases
        t = tables["tiny"]
        s0, s1 = t.rec_seg_off[r], t.rec_seg_off[r + 1]
        assert (t.seg_end[s0:s1] - t.seg_start[s0:s1] + 1).sum() <= 2
    assert len(want["small"][0]) <= 32768 and len(want["exon"][0]) > 100 * 32768
    return tables, want


PAIRS = [("exon", "cds"), ("small", "exon"), ("exon", "small"), ("cds", "cds"), ("empty", "cds"), ("exon", "tiny")]
OUTPUTS = [(a, bn, bp) for a in (0, 1) for bn in (0, 1) for bp in (0, 1)]        # (0, 0, 0): all NULL


@pytest.mark.parametrize("prep", ["prepare", "async_loose", "async_tight"])
@pytest.mark.parametrize("pair", PAIRS, ids=["%s-%s" % p for p in PAIRS])
def test_products_matrix(twin, products, tune, pair, prep):
    import torch
    from magot_b200 import _lib
    tables, want = products
    L, s = lib(), twin.streams[0]
    ka, kb = pair
    pa = twin.plan(ka, tables[ka])
    pb = pa if kb == ka else twin.plan(kb, tables[kb])
    wa, wb = want[ka], want[kb]

    def caps(p, w):                                       # prepare: the buffers hold the texts exactly
        if prep != "async_loose":
            return len(w[0]), len(w[1])
        c = p.capacities()
        return c[0] + 4096, c[1] + 4096

    ca, cb = caps(pa, wa), caps(pb, wb)
    out = {"a": new_buf(ca[0], s), "bn": new_buf(cb[0], s), "bp": new_buf(cb[1], s)}
    for lag in LAGS:
        tune("multi_lag", lag)
        for sel in OUTPUTS:
            for p, c in ((pa, ca), (pb, cb)) if pb is not pa else ((pa, ca),):
                if prep == "prepare":
                    p.prepare()
                else:
                    chk(L.mg_plan_prepare_async(p.handle, _lib.MG_PROT_TRIMX, c[0], c[1], sp(s)))
            poison(out.values(), twin.streams[0])
            oa, obn, obp = (out[k] if on else None for k, on in zip(("a", "bn", "bp"), sel))
            chk(L.mg_emit_products_device(pa.handle, P(oa), pb.handle, P(obn), P(obp), sp(s)))
            if sel == (0, 0, 0):
                chk(L.mg_emit_products_device(None, None, None, None, None, sp(s)))
            torch.cuda.synchronize()
            what = "%s lag %d outputs %s" % (prep, lag, sel)
            check_text(out["a"], wa[0] if sel[0] else None, what + " a")
            check_text(out["bn"], wb[0] if sel[1] else None, what + " b nucleotide")
            check_text(out["bp"], wb[1] if sel[2] else None, what + " b protein")
            assert pa.totals() == (len(wa[0]), len(wa[1])) and pb.totals() == (len(wb[0]), len(wb[1])), what
    torch.cuda.synchronize()
    pa.close()
    if pb is not pa:
        pb.close()


@pytest.mark.parametrize("short", ["a", "bn", "bp"])
def test_products_capacity_truncation(twin, products, short):
    """A capacity below the real size: mg_plan_totals reports it, the text is cut at the capacity, and nothing is written
    more than one 32-byte store plus its 32 bytes of padding (64 bytes) past the capacity."""
    import torch
    from magot_b200 import _lib
    tables, want = products
    L, s = lib(), twin.streams[0]
    pa, pb = twin.plan("exon"), twin.plan("cds")
    wa, wb = want["exon"], want["cds"]
    ca, cb = [len(wa[0]), len(wa[1])], [len(wb[0]), len(wb[1])]
    short_cap = {"a": (ca, 0), "bn": (cb, 0), "bp": (cb, 1)}[short]
    short_cap[0][short_cap[1]] -= 40_000
    out = {"a": new_buf(len(wa[0]), s), "bn": new_buf(len(wb[0]), s), "bp": new_buf(len(wb[1]), s)}
    poison(out.values(), twin.streams[0])
    chk(L.mg_plan_prepare_async(pa.handle, _lib.MG_PROT_TRIMX, ca[0], ca[1], sp(s)))
    chk(L.mg_plan_prepare_async(pb.handle, _lib.MG_PROT_TRIMX, cb[0], cb[1], sp(s)))
    chk(L.mg_emit_products_device(pa.handle, P(out["a"]), pb.handle, P(out["bn"]), P(out["bp"]), sp(s)))
    torch.cuda.synchronize()
    bad = pa if short == "a" else pb
    with pytest.raises(_lib.MagotError):
        bad.totals()
    for k, w, cap in (("a", wa[0], ca[0]), ("bn", wb[0], cb[0]), ("bp", wb[1], cb[1])):
        got = out[k].cpu().numpy()
        if k != short:
            check_text(out[k], w, k)
            continue
        assert cap < len(w)
        assert got[:cap].tobytes() == w[:cap], k
        beyond = np.flatnonzero(got[cap + 64:] != POISON)
        assert beyond.size == 0, "%s: byte %d written past the capacity %d" % (k, cap + 64 + beyond[0], cap)
    pa.close()
    pb.close()
