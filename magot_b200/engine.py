"""Host-side plumbing between the Python API (magot_b200.genome) and the C ABI.

`DeviceGenome`  -- one packed, device-resident genome replica (mg_genome handle).
`RecordTable`   -- the SoA interval tables the host flattener produces (contig id, start, end,
                   strand per segment, sorted per transcript in reference emission order, plus the
                   literal framing of each FASTA record).
`run_table`     -- create a plan, prepare (clamp + scans on the device), emit, copy back.
`ShardedGenome` -- replicas on several GPUs of one box; records are split into contiguous,
                   byte-balanced batches, one per GPU, and the texts are concatenated on the host
                   in record order (the path has no cross-shard reduction, hence no NCCL).

PyTorch is used only to obtain pinned host buffers; everything else is ctypes + numpy.
"""
import ctypes
import threading

import numpy as np

from . import _lib
from ._lib import lib, check
from .tables import RecordTable  # noqa: F401  (re-exported: engine.RecordTable)

_CHUNK = 64 << 20          # bases per mg_genome_pack call (multiple of 32)

#: mg_cds_check (include/magot_b200.h) as a numpy record: the per-record result of Plan.check
CHECK_DTYPE = np.dtype([("nuc_len", np.int64), ("gc", np.int64), ("n_codons", np.int32), ("n_ambig", np.int32),
                        ("n_stop", np.int32), ("first_stop", np.int32), ("gc3", np.int32), ("n_junction", np.int32),
                        ("n_noncanonical", np.int32), ("flags", np.int32), ("skip", np.int8), ("rem", np.int8),
                        ("start_codon", np.uint8), ("stop_codon", np.uint8), ("pad", np.int32)])
assert CHECK_DTYPE.itemsize == ctypes.sizeof(_lib.MgCdsCheck)

#: mg_cds_pred (include/magot_b200.h): the per-record result of Plan.predict_cds
PRED_DTYPE = np.dtype([("lo", np.int64), ("hi", np.int64), ("n_aa", np.int32), ("frame", np.int8), ("type", np.int8),
                       ("start_codon", np.uint8), ("stop_codon", np.uint8), ("n_cds_seg", np.int32), ("pad", np.int32)])
assert PRED_DTYPE.itemsize == ctypes.sizeof(_lib.MgCdsPred)

#: mg_cds_seg: each caller segment's share of its record's predicted CDS (-1, -1, -1 = empty)
CDSSEG_DTYPE = np.dtype([("lo", np.int64), ("hi", np.int64), ("phase", np.int8), ("pad", np.int8, (7,))])
assert CDSSEG_DTYPE.itemsize == ctypes.sizeof(_lib.MgCdsSeg)

#: mg_var_effect (include/magot_b200.h): one row of Plan.variant_effects
VEF_DTYPE = np.dtype([("var", np.int64), ("rec", np.int64), ("seg", np.int64), ("nuc_lo", np.int64), ("nuc_hi", np.int64),
                      ("codon", np.int32), ("cls", np.int8), ("n_aff", np.int8), ("ref_codon", np.uint8),
                      ("alt_codon", np.uint8), ("ref_aa", "S8"), ("alt_aa", "S8")])
assert VEF_DTYPE.itemsize == ctypes.sizeof(_lib.MgVarEffect)


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data) if a is not None else None


def pinned_empty(nbytes):
    """uint8 host buffer of nbytes, page-locked when torch + CUDA are available (plumbing only)."""
    try:
        import torch
        if torch.cuda.is_available():
            t = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, pin_memory=True)
            return t.numpy()[:nbytes]          # the ndarray keeps the tensor's storage alive
    except Exception:
        pass
    return np.empty(nbytes, dtype=np.uint8)


_PyBytes_New = ctypes.pythonapi.PyBytes_FromStringAndSize
_PyBytes_New.restype = ctypes.py_object
_PyBytes_New.argtypes = [ctypes.c_char_p, ctypes.c_ssize_t]
_PyBytes_Buf = ctypes.pythonapi.PyBytes_AsString
_PyBytes_Buf.restype = ctypes.c_void_p
_PyBytes_Buf.argtypes = [ctypes.py_object]


def new_bytes(n):
    """(bytes object of n uninitialised bytes, address of its buffer): the library writes the text straight into the object
    the API returns (CPython's own way of building a bytes result), no bytearray / numpy detour."""
    obj = _PyBytes_New(None, int(n))
    return obj, _PyBytes_Buf(obj)


def decode_text(text, strip_last=0):
    """latin-1 str of a bytes text without its last `strip_last` bytes (no intermediate bytes copy)."""
    if strip_last:
        return str(memoryview(text)[:len(text) - strip_last], "latin-1")
    return text.decode("latin-1")


class DeviceGenome(object):
    """A genome replica on one CUDA device: nibble-packed contigs + exception side list."""

    def __init__(self, contig_lens, device=0):
        _lib.require_device(device)
        self.device = device
        self.lens = np.ascontiguousarray(contig_lens, dtype=np.int64)
        self.handle = ctypes.c_void_p()
        check(lib.mg_genome_create(device, len(self.lens), _ptr(self.lens), ctypes.byref(self.handle)))
        self.n_exceptions = None

    def pack(self, contig, ascii_arr, offset=0):
        """Pack a uint8 array of FASTA bytes (newlines removed) into contig `contig` at `offset`."""
        a = np.ascontiguousarray(ascii_arr, dtype=np.uint8)
        n = a.size
        done = 0
        while done < n or (n == 0 and done == 0):
            m = min(_CHUNK, n - done)
            check(lib.mg_genome_pack(self.handle, contig, offset + done, ctypes.c_void_p(a.ctypes.data + done), m, None))
            done += m
            if n == 0:
                break

    def pack_fasta(self, contig, raw, lo=0, hi=None):
        """Pack contig `contig` from the RAW body of its FASTA record, raw[lo:hi] (bytes / uint8 array, line ends
        included): CR and LF are removed on the device (K0f), the host does not copy or scan the bases."""
        a = raw if isinstance(raw, np.ndarray) else np.frombuffer(raw, dtype=np.uint8)
        hi = a.size if hi is None else hi
        check(lib.mg_genome_pack_fasta(self.handle, contig, ctypes.c_void_p(a.ctypes.data + lo), hi - lo, None))

    def pack_device(self, contig, dev_ptr, n, offset=0, stream=None):
        check(lib.mg_genome_pack_device(self.handle, contig, offset, ctypes.c_void_p(dev_ptr), n, stream))

    def finalize(self):
        n = ctypes.c_int64(0)
        check(lib.mg_genome_finalize(self.handle, ctypes.byref(n)))
        self.n_exceptions = n.value
        return n.value

    def fetch(self, contig, lo, hi, minus=False):
        """Exact FASTA bytes of contig[lo:hi] (already clamped), or their reverse complement."""
        n = hi - lo
        if n <= 0:
            return b""
        out = np.empty(n, dtype=np.uint8)
        check(lib.mg_genome_fetch(self.handle, contig, lo, hi, 1 if minus else 0, _ptr(out), None))
        return out.tobytes()

    def mask(self, contig, lo, hi, hard=False, upper_first=False):
        """K5: lower-case (soft) or 'N' (hard) the 0-based half-open intervals, optionally upper-casing everything first."""
        contig = np.ascontiguousarray(contig, dtype=np.int32)
        lo = np.ascontiguousarray(lo, dtype=np.int64)
        hi = np.ascontiguousarray(hi, dtype=np.int64)
        check(lib.mg_genome_mask(self.handle, contig.size, _ptr(contig), _ptr(lo), _ptr(hi), int(bool(hard)), int(bool(upper_first)), None))

    def device_bytes(self):
        return lib.mg_genome_bytes(self.handle)

    def close(self):
        if self.handle:
            lib.mg_genome_destroy(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Plan(object):
    """mg_plan wrapper: create -> prepare -> emit."""

    def __init__(self, genome, table, stream=None):
        self.genome = genome
        self.table = table                       # keeps the host arrays alive
        self.stream = stream
        self.handle = ctypes.c_void_p()
        t = table
        check(lib.mg_plan_create(genome.handle, t.n_rec, _ptr(t.rec_seg_off), t.n_seg, _ptr(t.seg_contig),
                                 _ptr(t.seg_start), _ptr(t.seg_end), _ptr(t.seg_strand), _ptr(t.rec_lit_off),
                                 _ptr(t.rec_pre_len), _ptr(t.rec_suf_len), _ptr(t.lit), t.lit.size,
                                 _ptr(t.rec_phase), stream, ctypes.byref(self.handle)))
        self.nuc_total = None
        self.prot_total = None

    def set_codon_table(self, codon64):
        """Genetic code of this plan's protein text (mg_plan_set_codon_table): codon64 = 64 bytes as gencode.codon64(n),
        None = the standard code.  Takes effect for every emit queued after the call."""
        if codon64 is not None:
            codon64 = bytes(codon64)
            if len(codon64) != 64:
                raise ValueError("codon64 must hold 64 bytes")
        check(lib.mg_plan_set_codon_table(self.handle, codon64))

    def prepare(self, trimx=True, use_phase=False):
        flags = (_lib.MG_PROT_TRIMX if trimx else 0) | (_lib.MG_PROT_USE_PHASE if use_phase else 0)
        a, b = ctypes.c_int64(0), ctypes.c_int64(0)
        check(lib.mg_plan_prepare(self.handle, flags, ctypes.byref(a), ctypes.byref(b), self.stream))
        self.nuc_total, self.prot_total = a.value, b.value
        return self.nuc_total, self.prot_total

    def capacities(self):
        """Upper bounds of the two text sizes from the host tables alone (what mg_plan_prepare_async needs): every
        segment at most end-start+1 bases before clamping, a protein at most a third of its record's bases."""
        t = self.table
        pay = t.approx_bytes_per_record() - t.rec_pre_len - t.rec_suf_len
        lit = int(t.rec_pre_len.astype(np.int64).sum() + t.rec_suf_len.astype(np.int64).sum())
        return int(pay.sum()) + lit, int((pay // 3).sum()) + lit

    def prepare_async(self, nuc_capacity=None, prot_capacity=None, trimx=True, use_phase=False, defer_records=False):
        """K1 without the host round trip; sizes come later from totals().  defer_records: only the piece pass (what the
        nucleotide text needs); prepare_prot() runs the record pass before anything protein-related."""
        if nuc_capacity is None or prot_capacity is None:
            a, b = self.capacities()
            nuc_capacity = a if nuc_capacity is None else nuc_capacity
            prot_capacity = b if prot_capacity is None else prot_capacity
        flags = (_lib.MG_PROT_TRIMX if trimx else 0) | (_lib.MG_PROT_USE_PHASE if use_phase else 0) | (_lib.MG_PROT_DEFER if defer_records else 0)
        check(lib.mg_plan_prepare_async(self.handle, flags, int(nuc_capacity), int(prot_capacity), self.stream))
        self.nuc_total = self.prot_total = None
        return int(nuc_capacity), int(prot_capacity)

    def prepare_prot(self, stream=None):
        """The record pass a prepare_async(defer_records=True) left out (mg_plan_prepare_prot_async)."""
        check(lib.mg_plan_prepare_prot_async(self.handle, stream if stream is not None else self.stream))

    def totals(self):
        a, b = ctypes.c_int64(0), ctypes.c_int64(0)
        check(lib.mg_plan_totals(self.handle, ctypes.byref(a), ctypes.byref(b), self.stream))
        self.nuc_total, self.prot_total = a.value, b.value
        return self.nuc_total, self.prot_total

    def lengths(self):
        n = self.table.n_rec
        nuc = np.empty(n, dtype=np.int64)
        aa = np.empty(n, dtype=np.int64)
        check(lib.mg_plan_lengths(self.handle, _ptr(nuc), _ptr(aa), self.stream))
        return nuc, aa

    def check(self, start_codons=None, use_phase=False, codon_usage=False, junctions=False):
        """Gene-model check of every record (mg_plan_check) under the plan's genetic code.  start_codons: 64 flags as
        gencode.start64 gives them, None = ATG.  Returns (CHECK_DTYPE records, uint32 [n_rec, 64] codon counts or None,
        int8 junction class per segment of the table or None).  Needs prepare() or prepare_async() first."""
        n = self.table.n_rec
        recs = np.zeros(n, dtype=CHECK_DTYPE)
        counts = np.zeros((n, 64), dtype=np.uint32) if codon_usage else None
        junc = np.zeros(self.table.n_seg, dtype=np.int8) if junctions else None
        if start_codons is not None:
            start_codons = bytes(start_codons)
            if len(start_codons) != 64:
                raise ValueError("start_codons must hold 64 flags")
        check(lib.mg_plan_check(self.handle, _lib.MG_PROT_USE_PHASE if use_phase else 0, start_codons, _ptr(recs),
                                _ptr(counts), _ptr(junc), self.stream))
        check(lib.mg_stream_sync(self.genome.device, self.stream))
        return recs, counts, junc

    def predict_cds(self, min_aa, start_codons=None, partial5=False, partial3=False):
        """Longest ORF of every record (mg_plan_predict_cds) under the plan's genetic code.  start_codons: 64 flags as
        gencode.start64 gives them, None = ATG; partial5 / partial3: also ORFs open at the frame's 5' end / without a stop.
        Returns (PRED_DTYPE records, CDSSEG_DTYPE entry per segment of the table).  Needs prepare() or prepare_async() first."""
        recs = np.zeros(self.table.n_rec, dtype=PRED_DTYPE)
        segs = np.zeros(self.table.n_seg, dtype=CDSSEG_DTYPE)
        if start_codons is not None:
            start_codons = bytes(start_codons)
            if len(start_codons) != 64:
                raise ValueError("start_codons must hold 64 flags")
        flags = (_lib.MG_PRED_5PARTIAL if partial5 else 0) | (_lib.MG_PRED_3PARTIAL if partial3 else 0)
        check(lib.mg_plan_predict_cds(self.handle, int(min_aa), start_codons, flags, _ptr(recs), _ptr(segs), self.stream))
        check(lib.mg_stream_sync(self.genome.device, self.stream))
        return recs, segs

    def variant_effects(self, contig, pos, allele_off, allele_bytes, start_codons=None, use_phase=False):
        """Coding consequences of sorted alleles on every record (mg_plan_variant_count + mg_plan_variant_emit) under the plan's
        genetic code.  contig (int32), pos (int64, 0-based) per allele, sorted by (contig, pos); REF of allele i is
        allele_bytes[allele_off[2i]:allele_off[2i+1]], ALT the bytes up to allele_off[2i+2].  start_codons: 64 flags as
        gencode.start64 gives them, None = ATG.  Returns (int8 status per allele, VEF_DTYPE rows ordered by record, then
        allele).  Needs prepare() or prepare_async() first."""
        contig = np.ascontiguousarray(contig, dtype=np.int32)
        pos = np.ascontiguousarray(pos, dtype=np.int64)
        allele_off = np.ascontiguousarray(allele_off, dtype=np.int64)
        buf = np.frombuffer(bytes(allele_bytes), dtype=np.uint8) if not isinstance(allele_bytes, np.ndarray) else \
            np.ascontiguousarray(allele_bytes, dtype=np.uint8)
        n = contig.size
        if pos.size != n or allele_off.size != 2 * n + 1:
            raise ValueError("contig and pos need one entry per allele, allele_off 2 * n + 1")
        if start_codons is not None:
            start_codons = bytes(start_codons)
            if len(start_codons) != 64:
                raise ValueError("start_codons must hold 64 flags")
        status = np.zeros(n, dtype=np.int8)
        n_rows = ctypes.c_int64(0)
        check(lib.mg_plan_variant_count(self.handle, n, _ptr(contig), _ptr(pos), _ptr(allele_off), _ptr(buf), buf.size,
                                        _lib.MG_PROT_USE_PHASE if use_phase else 0, start_codons, _ptr(status),
                                        ctypes.byref(n_rows), self.stream))
        rows = np.zeros(n_rows.value, dtype=VEF_DTYPE)
        check(lib.mg_plan_variant_emit(self.handle, _ptr(rows), self.stream))
        check(lib.mg_stream_sync(self.genome.device, self.stream))
        return status, rows

    def emit_host(self, protein=False, out=None):
        total = self.prot_total if protein else self.nuc_total
        if out is None:
            out = np.empty(total, dtype=np.uint8)
        if total:
            fn = lib.mg_emit_prot_host if protein else lib.mg_emit_nuc_host
            check(fn(self.handle, _ptr(out), self.stream))
            check(lib.mg_stream_sync(self.genome.device, self.stream))
        return out[:total]

    def emit_bytes(self, protein=False):
        """The text as a bytes object, filled by the library (mg_emit_*_host: device text -> two page-locked staging buffers
        -> this object, pipelined)."""
        total = self.prot_total if protein else self.nuc_total
        if not total:
            return b""
        obj, addr = new_bytes(total)
        fn = lib.mg_emit_prot_host if protein else lib.mg_emit_nuc_host
        check(fn(self.handle, ctypes.c_void_p(addr), self.stream))
        check(lib.mg_stream_sync(self.genome.device, self.stream))
        return obj

    def emit_both_host(self):
        """K23 (mg_emit_nuc_prot_host): the nucleotide text and its translation from ONE pass over the genome, as the
        reference produces them (genome.py:704-707).  Returns (nuc, prot) uint8 arrays."""
        nuc = np.empty(self.nuc_total, dtype=np.uint8)
        prot = np.empty(self.prot_total, dtype=np.uint8)
        if self.nuc_total or self.prot_total:
            check(lib.mg_emit_nuc_prot_host(self.handle, _ptr(nuc), _ptr(prot), self.stream))
            check(lib.mg_stream_sync(self.genome.device, self.stream))
        return nuc, prot

    def emit_device(self, dev_ptr, protein=False):
        fn = lib.mg_emit_prot_device if protein else lib.mg_emit_nuc_device
        check(fn(self.handle, ctypes.c_void_p(dev_ptr), self.stream))

    def close(self):
        if self.handle:
            lib.mg_plan_destroy(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def run_table(genome, table, protein=False, trimx=True, use_phase=False, want_lengths=False, codon64=None):
    """One pass of the hot path over one batch on one GPU. Returns (text bytes, (nuc_len, aa_len) | None).
    codon64: genetic code of the protein text (gencode.codon64), None = the standard code."""
    plan = Plan(genome, table)
    try:
        if codon64 is not None:
            plan.set_codon_table(codon64)
        plan.prepare(trimx=trimx, use_phase=use_phase)
        lens = plan.lengths() if want_lengths else None
        text = plan.emit_bytes(protein=protein)
    finally:
        plan.close()
    return text, lens


def run_table_both(genome, table, trimx=True, use_phase=False, async_prepare=False, codon64=None):
    """Nucleotide AND protein text of one batch from one fused pass (K23). Returns (nuc bytes, prot bytes)."""
    plan = Plan(genome, table)
    try:
        if codon64 is not None:
            plan.set_codon_table(codon64)
        if async_prepare:
            plan.prepare_async(trimx=trimx, use_phase=use_phase)
            plan.totals()
        else:
            plan.prepare(trimx=trimx, use_phase=use_phase)
        nuc, prot = plan.emit_both_host()
    finally:
        plan.close()
    return nuc.tobytes(), prot.tobytes()


def run_products(genome, table_a, table_b, protein_b=True, trimx=True, use_phase=False, codon64=None):
    """mg_emit_products_host: nucleotide text of table_a, nucleotide (+ protein) text of table_b from one launch.
    Returns (text_a, nuc_b, prot_b) as bytes (prot_b is b"" without protein_b)."""
    pa, pb = Plan(genome, table_a), Plan(genome, table_b)
    try:
        if codon64 is not None:
            pb.set_codon_table(codon64)
        pa.prepare(trimx=trimx, use_phase=use_phase)
        pb.prepare(trimx=trimx, use_phase=use_phase)
        oa = np.empty(pa.nuc_total, dtype=np.uint8)
        obn = np.empty(pb.nuc_total, dtype=np.uint8)
        obp = np.empty(pb.prot_total if protein_b else 0, dtype=np.uint8)
        check(lib.mg_emit_products_host(pa.handle, _ptr(oa), pb.handle, _ptr(obn), _ptr(obp) if protein_b else None, None))
        check(lib.mg_stream_sync(genome.device, None))
    finally:
        pa.close()
        pb.close()
    return oa.tobytes(), obn.tobytes(), obp.tobytes()


def shard_bounds(weights, n_shards):
    """Split records into n_shards contiguous batches of ~equal total weight (prefix sum / n)."""
    n = len(weights)
    if n_shards <= 1 or n == 0:
        return [0, n]
    csum = np.cumsum(np.asarray(weights, dtype=np.float64))
    total = csum[-1] if n else 0.0
    bounds = [0]
    for k in range(1, n_shards):
        target = total * k / n_shards
        bounds.append(min(n, max(bounds[-1], int(np.searchsorted(csum, target, side="left")) + 1)))
    bounds.append(n)
    return bounds


class ShardedGenome(object):
    """The same packed genome replicated on several GPUs of one box."""

    def __init__(self, replicas):
        self.replicas = list(replicas)

    @property
    def primary(self):
        return self.replicas[0]

    def run_table(self, table, protein=False, trimx=True, use_phase=False, want_lengths=False, codon64=None):
        if len(self.replicas) == 1 or table.n_rec < 2 * len(self.replicas):
            return run_table(self.primary, table, protein, trimx, use_phase, want_lengths, codon64)
        bounds = shard_bounds(table.approx_bytes_per_record(), len(self.replicas))
        results = [None] * len(self.replicas)
        errors = []

        def work(k):
            try:
                r0, r1 = bounds[k], bounds[k + 1]
                if r1 > r0:
                    results[k] = run_table(self.replicas[k], table.slice(r0, r1), protein, trimx, use_phase, want_lengths, codon64)
                else:
                    results[k] = (b"", (np.empty(0, np.int64), np.empty(0, np.int64)) if want_lengths else None)
            except Exception as e:      # re-raised on the caller's thread
                errors.append(e)

        threads = [threading.Thread(target=work, args=(k,)) for k in range(len(self.replicas))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        text = b"".join(r[0] for r in results)
        lens = None
        if want_lengths:
            lens = (np.concatenate([r[1][0] for r in results]), np.concatenate([r[1][1] for r in results]))
        return text, lens

    def close(self):
        for r in self.replicas:
            r.close()
