"""Start-to-stop ORF calling on the device (mg_orfcall_*, orfs.call_orfs, genome_tools call_orfs), bit-exact against the
numpy reference orfcall_ref: every scan variant, the dense second pass, contig lists in any order, five genetic codes, three
start sets, nine minimum lengths, with and without 3' partials; no interference with the six-frame scan; the config-5
genome at full size."""
import contextlib
import ctypes
import io

import numpy as np
import pytest

import gencode_ref as gref
import orfcall_ref as ref

pytestmark = pytest.mark.gpu

CODES = (1, 2, 6, 11, 23)
MIN_AA = (0, 1, 30, 47, 48, 95, 96, 100, 300)
SENSE = tuple(c for c in ("ACGT"[i >> 4] + "ACGT"[(i >> 2) & 3] + "ACGT"[i & 3] for i in range(64)))
START_SETS = (("ATG",), ("ATG", "GTG", "TTG"), "sense")


@pytest.fixture(scope="module")
def mg():
    import magot_b200
    return magot_b200


@pytest.fixture()
def six_mode(mg):
    from magot_b200 import _lib
    yield lambda v: _lib.check(_lib.lib.mg_tune(b"six", v))
    _lib.check(_lib.lib.mg_tune(b"six", 2))


def _genome(contigs):
    from magot_b200 import engine
    g = engine.DeviceGenome([len(c) for c in contigs], device=0)
    for i, c in enumerate(contigs):
        g.pack(i, np.frombuffer(c, dtype=np.uint8))
    g.finalize()
    return g


def _starts(code, which):
    if which != "sense":
        return which
    t = gref.table64(code)
    return tuple(c for c in SENSE if t[ref.codon_index(c)] != "*")


def _contigs(rng):
    alpha = np.frombuffer(b"ACGTACGTACGTacgtN", dtype=np.uint8)
    out = []
    for n in (0, 1, 2, 3, 4, 5, 6, 7, 8, 1000, 24575, 24576, 24577, 73727, 73728, 73729, 147455, 147457, 200001):
        out.append(alpha[rng.integers(0, alpha.size, size=n)].tobytes())
    ac = np.frombuffer(b"AC", dtype=np.uint8)                 # stop-poor: long stretches without a stop on the plus strand
    c = bytearray(alpha[rng.integers(0, 4, size=160000)].tobytes())
    c[20000:140000] = ac[rng.integers(0, 2, size=120000)].tobytes()
    for k in range(20000, 140000, 9001):
        c[k:k + 3] = b"ATG"
    out.append(bytes(c))
    c = bytearray(alpha[rng.integers(0, 4, size=80000)].tobytes())   # N runs
    c[1000:30000] = b"N" * 29000
    c[50000:50005] = b"NNNNN"
    out.append(bytes(c))
    # a start at the first codon and a stop at the last codon of every phase, on both strands
    for L in range(6, 16):
        for p in range(3):
            s = bytearray(np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=L)].tobytes())
            s[p:p + 3] = b"ATG"
            last = p + 3 * ((L - p) // 3 - 1)
            if last > p:
                s[last:last + 3] = b"TGA"
            out.append(bytes(s))
            out.append(gref.revcomp(bytes(s)))
    return out


def _got(recs, aa):
    rows = [tuple(int(v) for v in r) for r in recs[["contig", "minus", "phase", "flags", "start_codon", "lo", "hi", "len",
                                                     "aa_off"]].tolist()]
    return rows, aa


def _filtered(full, min_aa, partial):
    """The reference at (min_aa, partial) from its min_aa = 0, partial = True result: keep len >= min_aa and a stop, or
    partial; the residue offsets follow."""
    recs, aa = full
    out, parts, off = [], [], 0
    for r in recs:
        if r[7] >= min_aa and (r[3] == 0 or partial):
            out.append(r[:8] + (off,))
            parts.append(aa[r[8]:r[8] + r[7]])
            off += r[7]
    return out, b"".join(parts)


def test_orfcall_grid(mg, six_mode, monkeypatch):
    from magot_b200 import orfs
    rng = np.random.default_rng(11)
    contigs = _contigs(rng)
    n = len(contigs)
    g = _genome(contigs)
    ids = list(range(n))
    perm = [n - 1, 3, 20, 0, 18, 18, 12, 21, 5]
    try:
        for code in CODES:
            for which in START_SETS:
                starts = _starts(code, which)
                full = ref.call_list(contigs, ids, 0, code, starts, True)
                full_perm = ref.call_list(contigs, perm, 0, code, starts, True)
                for min_aa in MIN_AA:
                    for partial in (False, True):
                        want = _filtered(full, min_aa, partial)
                        for mode in (2, 1, 0):
                            six_mode(mode)
                            got = _got(*orfs.call_orfs(g, ids, min_aa, code, starts, partial))
                            assert got == want, (code, which, min_aa, partial, mode)
                        six_mode(2)
                        got = _got(*orfs.call_orfs(g, perm, min_aa, code, starts, partial))
                        assert got == _filtered(full_perm, min_aa, partial), (code, which, min_aa, partial, "list")
        # the dense second pass: the hit list overflows, from the single-pass and the two-level scan
        monkeypatch.setenv("MG_SIX_HIT_CAP", "7")
        for code in (1, 23):
            starts = ("ATG", "GTG", "TTG")
            full = ref.call_list(contigs, ids, 0, code, starts, True)
            for min_aa in (0, 1, 30, 100):
                for partial in (False, True):
                    for mode in (2, 0):
                        six_mode(mode)
                        got = _got(*orfs.call_orfs(g, ids, min_aa, code, starts, partial))
                        assert got == _filtered(full, min_aa, partial), ("dense", code, min_aa, partial, mode)
    finally:
        g.close()


def test_orfcall_translation_consistency(mg):
    """The plan path's nucleotide text of each ORF with a stop, translated by Sequence.translate, is the protein with its
    first residue as coded and a final '*'."""
    from magot_b200 import engine, orfs
    rng = np.random.default_rng(12)
    contigs = [np.frombuffer(b"ACGTacgtN", dtype=np.uint8)[rng.integers(0, 9, size=n)].tobytes() for n in (50000, 9001, 30)]
    g = _genome(contigs)
    try:
        for code in (1, 2, 23):
            recs, aa = orfs.call_orfs(g, [0, 1, 2], 10, code, ("ATG", "GTG", "TTG", "CTG"), partial=True)
            R = recs.size
            assert R > 50
            zero = np.zeros(R, dtype=np.int32)
            tbl = engine.RecordTable(np.arange(R + 1), recs["contig"], recs["lo"] + 1, recs["hi"], recs["minus"],
                                     np.zeros(R, dtype=np.int64), zero, zero, np.zeros(0, dtype=np.uint8))
            text, (nuc_len, _) = engine.run_table(g, tbl, want_lengths=True)
            off = np.concatenate(([0], np.cumsum(nuc_len)))
            for k, r in enumerate(recs):
                nuc = text[off[k]:off[k + 1]].decode()
                prot = aa[int(r["aa_off"]):int(r["aa_off"]) + int(r["len"])].decode()
                assert prot[0] == "M"
                t = mg.Sequence(nuc).translate(genetic_code=code)
                if int(r["flags"]) & 1:
                    assert t[1:] == prot[1:]
                else:
                    assert t[1:] == prot[1:] + "*"
    finally:
        g.close()


def test_no_interference_with_sixframe(mg, six_mode):
    from magot_b200 import orfs, _lib
    rng = np.random.default_rng(13)
    contigs = [np.frombuffer(b"ACGTacgtN", dtype=np.uint8)[rng.integers(0, 9, size=n)].tobytes() for n in (300000, 73729, 5000)]
    g = _genome(contigs)
    lib = _lib.lib
    try:
        six_mode(2)
        before = {code: orfs.sixframe(g, 0, 3, 100, genetic_code=code) for code in (1, 2)}
        same = lambda a, b: a[1] == b[1] and np.array_equal(a[0], b[0])   # noqa: E731
        # the standard stop index is built by now: the same call launches as many kernels after an ORF call as before it
        k0 = lib.mg_kernel_launches()
        assert same(orfs.sixframe(g, 0, 3, 100), before[1])
        per_call = lib.mg_kernel_launches() - k0
        for code in (1, 2):
            orfs.call_orfs(g, [0, 1, 2], 100, code)
            orfs.call_orfs(g, [2, 0], 30, code, ("ATG", "TTG"), partial=True)
            k0 = lib.mg_kernel_launches()
            assert same(orfs.sixframe(g, 0, 3, 100), before[1])
            assert lib.mg_kernel_launches() - k0 == per_call, "the standard stop index was rebuilt"
            assert same(orfs.sixframe(g, 0, 3, 100, genetic_code=2), before[2])
        # mismatched emits
        ids = np.arange(3, dtype=np.int64)
        n_orf, n_bytes = ctypes.c_int64(0), ctypes.c_int64(0)
        recs = (_lib.MgOrfCall * 1)()
        _lib.check(lib.mg_sixframe_count(g.handle, 0, 3, 100, ctypes.byref(n_orf), ctypes.byref(n_bytes), None))
        assert lib.mg_orfcall_emit(g.handle, None, recs, None) == -4
        assert "mg_orfcall_count" in _lib.last_error()
        _lib.check(lib.mg_orfcall_count(g.handle, 3, ctypes.c_void_p(ids.ctypes.data), 100, None, None, 0, ctypes.byref(n_orf),
                                        ctypes.byref(n_bytes), None))
        assert lib.mg_sixframe_emit(g.handle, None, recs, None) == -4
        assert "mg_sixframe_count" in _lib.last_error()
        assert lib.mg_sixframe_emit_device(g.handle, None, None, None) == -4
        # argument checks of the C entry point
        none = bytes(64)
        taa = bytearray(64)
        taa[ref.codon_index("TAA")] = 1
        for start64 in (none, bytes(taa)):
            assert lib.mg_orfcall_count(g.handle, 3, ctypes.c_void_p(ids.ctypes.data), 100, None, start64, 0, ctypes.byref(n_orf),
                                        ctypes.byref(n_bytes), None) == -1
    finally:
        g.close()


def _stdout_of(fn, *a, **k):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        fn(*a, **k)
    return buf.getvalue()


@pytest.mark.parametrize("out_format", ["gff3", "protein", "nucleotide"])
def test_call_orfs_cli(mg, tmp_path, out_format):
    from magot_b200 import genome_tools as gt
    import py2dict
    rng = np.random.default_rng(14)
    seqs = {"s1": rng.choice(list("ACGT"), size=2000), "s2 x": rng.choice(list("ACGTNacgt"), size=7001),
            "s3": rng.choice(list("ACGT"), size=4), "chr9": rng.choice(list("ACGT"), size=30000)}
    seqs = {k: "".join(v) for k, v in seqs.items()}
    fa = tmp_path / "g.fa"
    fa.write_text("".join(">%s\n%s\n" % kv for kv in seqs.items()))
    order = py2dict.py2_order(list(seqs))
    contigs = [seqs[k].encode() for k in order]
    names = {i: k for i, k in enumerate(order)}
    for code, starts, min_orf, partial in ((11, "ATG,GTG,TTG", 30, "False"), (1, "ATG", 100, "True"), (2, "ATG,atg,ATA", 0, "True")):
        got = _stdout_of(gt.call_orfs, str(fa), min_orf=str(min_orf), genetic_code=str(code), start_codons=starts,
                         partial=partial, out_format=out_format)
        want = ref.cli_lines(contigs, names, range(len(order)), min_orf, code, starts.upper().split(","), partial == "True",
                             out_format)
        assert got == "\n".join(want) + ("\n" if want else "")
    # the FUNCTIONS table and the command-line grammar
    got = _stdout_of(gt.main, ["genome_tools", "call_orfs", str(fa), "min_orf=100", "genetic_code=11", "start_codons=ATG,GTG,TTG"])
    want = ref.cli_lines(contigs, names, range(len(order)), 100, 11, ["ATG", "GTG", "TTG"], False, "gff3")
    assert got == "\n".join(want) + "\n"


# ---- full size ----------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def big():
    """BASELINE config 5: the 3.1 Gbp genome in 24 chromosomes + 170 scaffolds, built as test_gpu_fullsize.py builds it."""
    import torch
    from magot_b200 import engine, synth, _lib
    _lib.require_device(0)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    layout = synth.contig_layout("human", 3_100_000_000, 4)
    g = engine.DeviceGenome([l for _, l in layout], device=0)
    CH = 256 << 20
    host = []
    for ci, (_, L) in enumerate(layout):
        h = np.empty(L, dtype=np.uint8)
        for off in range(0, L, CH):
            n = min(CH, L - off)
            a = synth.synth_contig_device(n, 4 * 1000003 + ci * 64 + off // CH, dev)
            h[off:off + n] = a.cpu().numpy()
            g.pack_device(ci, a.data_ptr(), n, offset=off)
            torch.cuda.synchronize()
            del a
        host.append(h)
    g.finalize()
    torch.cuda.empty_cache()
    yield g, layout, host
    g.close()


def test_config5_orfcall_full_size(big):
    from magot_b200 import orfs
    g, layout, host = big
    ids = list(range(len(layout)))
    recs, aa = orfs.call_orfs(g, ids, 100)
    assert recs.size > 10_000
    assert int(recs["len"].min()) >= 100
    a = np.frombuffer(aa, dtype=np.uint8)
    assert a.size == int(recs["len"].sum())
    assert not (a == ord("*")).any()
    assert (a[recs["aa_off"]] == ord("M")).all()
    assert (recs["flags"] == 0).all()
    # the list split at an arbitrary point gives the same records and residues
    cut = 57
    r1, a1 = orfs.call_orfs(g, ids[:cut], 100)
    r2, a2 = orfs.call_orfs(g, ids[cut:], 100)
    assert a1 + a2 == aa
    both = np.concatenate((r1, r2))
    both["aa_off"][r1.size:] += len(a1)
    assert np.array_equal(both, recs)
    # the scaffolds and the smallest chromosome against the reference on the host copy of the bases
    lens = [l for _, l in layout]
    chrom = int(np.argmin(lens[:24]))
    sub = [chrom] + list(range(24, len(layout)))
    got = orfs.call_orfs(g, sub, 100)
    want = ref.call_list({c: host[c].tobytes() for c in sub}, sub, 100)
    assert _got(*got) == want
