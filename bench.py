#!/usr/bin/env python3
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py ... --dump-outputs DIR                   (what the last timed step computed, as DIR/*.npy)

Workload (config.workload): synthetic 3.1 Gbp human-scale genome (24 chromosomes + 170 scaffolds,
5 % N, 50 % soft-masked) resident on the GPU as two strand planes of 0.5 B/base each, and a GTF-shaped annotation of 200k
transcripts per GPU (weak scaling: every rank owns its own 200k-transcript batch over a replicated
genome; the path has no cross-shard exchange, so there is no collective on the data path).
One STEP = one pass of the hot path over one batch, producing all three products of config 4:
CDS nucleotide FASTA, CDS protein FASTA, exon-based transcript FASTA (K1 clamp+scan, K2 splice+RC,
K3 translate, FASTA framing on the device).
metric  spliced+translated Gbp/s = (CDS bp spliced + CDS bp translated + exon bp spliced) / time.
value   device-resident: interval tables already in HBM, outputs left in HBM (CUDA events).
e2e     through the C ABI with HOST buffers: pinned SoA tables -> H2D -> kernels -> D2H of the three
        texts into pinned memory, every step.
The reference arm (--impl reference) times the reference's own Python get_fasta (oracle/_ref, the shimmed
reference; else the oracle port) on the host cores on a bounded sample of the same workload shape.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GENOME_BP = int(os.environ.get("MAGOT_BENCH_GENOME_BP", 3_100_000_000))
N_TX = int(os.environ.get("MAGOT_BENCH_TX", 200_000))
SAMPLE_BP = int(os.environ.get("MAGOT_BENCH_SAMPLE_BP", 20_000_000))
SAMPLE_TX = int(os.environ.get("MAGOT_BENCH_SAMPLE_TX", 1290))
SEED = 4
METRIC = "spliced+translated Gbp/s"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return float(p["hbm_gbs"]), "MEASURED_PEAKS.json (measured copy bandwidth)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# CPU legs (rank 0 only): the reference's own code on a bounded sample
# ------------------------------------------------------------------------------------------------------
def build_sample():
    """Scaled twin of the workload (same generators): host genome + annotation + GTF text."""
    from magot_b200 import synth
    layout = synth.contig_layout("human", SAMPLE_BP, SEED)
    contigs = synth.synth_genome_host(layout, SEED)
    ann = synth.synth_annotation(layout, SAMPLE_TX, SEED)
    return layout, contigs, ann


def _sample_bp(ann):
    return 2 * ann.spliced_bp("cds") + ann.spliced_bp("exon")


_REF_STATE = {}


def _ref_worker(args):
    which, seq_type, keys = args
    g = _REF_STATE[which]
    n = 0
    for k in keys:
        n += len(g.annotations.gene[k].get_fasta(seq_type=seq_type))
    return n


def reference_setup(layout, contigs, ann):
    """Build the reference's (or the port's) objects for the sample. Returns (kind, run_step(pool) -> bytes)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    names = [n for n, _ in layout]
    fasta = "".join(">%s\n%s\n" % (n, c.tobytes().decode("latin-1")) for n, c in zip(names, contigs))
    try:
        import ref_runner
        ref = ref_runner.ref()
    except Exception:
        ref = None
    if ref is not None:
        kind = "reference"
        # The reference's own classes, populated directly (what its read_gff builds for a GTF: gene ->
        # transcript -> CDS|exon); read_gff itself costs ~1 ms/line in the reference and is not the timed path.
        for which in ("cds", "exon"):
            gs = ref.GenomeSequence(fasta)
            g = ref.Genome(gs)
            aset = ref.AnnotationSet()
            aset.genome = g
            g.annotations = aset
            off, st, en = (ann.cds_off, ann.cds_start, ann.cds_end) if which == "cds" else (ann.exon_off, ann.exon_start, ann.exon_end)
            ftype = "CDS" if which == "cds" else "exon"
            if ftype not in aset.__dict__:
                aset.__dict__[ftype] = {}
            for t in range(ann.n_tx):
                tx = ann.names[t]
                gid = "g%d" % ann.gene_of[t]
                ctg = names[ann.contig[t]]
                sd = "-" if ann.strand[t] else "+"
                if gid not in aset.gene:
                    aset.gene[gid] = ref.ParentAnnotation(gid, ctg, "gene", [], None, sd, aset)
                aset.gene[gid].child_list.append(tx)
                kids = []
                for k in range(off[t], off[t + 1]):
                    cid = "%s-%s%d" % (tx, ftype, k - off[t])
                    kids.append(cid)
                    aset.__dict__[ftype][cid] = ref.BaseAnnotation(cid, ctg, (int(st[k]), int(en[k])), ftype, tx, sd, {}, aset)
                aset.transcript[tx] = ref.ParentAnnotation(tx, ctg, "transcript", kids, gid, sd, aset)
            _REF_STATE[which] = g
        keys = list(_REF_STATE["cds"].annotations.gene)
    else:
        kind = "port"
        import magot_oracle as mo
        gtf = ann.to_gtf(names)
        seqs, _ = mo.read_fasta(fasta)

        class _G(object):
            pass
        for which, kw in (("cds", {}), ("exon", {"base_features": ('exon', 'match_part', 'similarity', 'region'), "features_to_ignore": ('CDS',)})):
            aset = mo.read_gff(gtf, **kw)
            aset.genome = seqs
            g = _G()
            g.annotations = _G()

            class _Wrap(object):
                def __init__(self, o):
                    self.o = o

                def get_fasta(self, seq_type="nucleotide"):
                    return mo.parent_get_fasta(self.o, seq_type=seq_type)
            g.annotations.gene = {k: _Wrap(v) for k, v in aset.table('gene').items()}
            _REF_STATE[which] = g
        keys = list(_REF_STATE["cds"].annotations.gene)
    return kind, keys


def reference_step(pool, keys, workers):
    tasks = []
    for which, seq_type in (("cds", "nucleotide"), ("cds", "protein"), ("exon", "nucleotide")):
        chunk = max(1, (len(keys) + workers * 4 - 1) // (workers * 4))
        for i in range(0, len(keys), chunk):
            tasks.append((which, seq_type, keys[i:i + chunk]))
    if pool is None:
        return sum(_ref_worker(t) for t in tasks)
    return sum(pool.map(_ref_worker, tasks))


def cpu_reference_rate(steps, warmup, workers):
    """Gbp/s of the reference's get_fasta path on the sample with `workers` processes."""
    import multiprocessing as mp
    layout, contigs, ann = build_sample()
    kind, keys = reference_setup(layout, contigs, ann)
    bp = _sample_bp(ann)
    pool = mp.get_context("fork").Pool(workers) if workers > 1 else None
    try:
        for _ in range(warmup):
            reference_step(pool, keys, workers)
        t0 = time.perf_counter()
        for _ in range(steps):
            reference_step(pool, keys, workers)
        dt = (time.perf_counter() - t0) / max(steps, 1)
    finally:
        if pool is not None:
            pool.terminate()
    sample = "config-4 generators at 1/%d scale: %d bp genome, %d transcripts, CDS nuc + CDS protein + exon transcripts via get_fasta (%s, CPython %d.%d; Python 2.7 is not available)" % (
        max(1, GENOME_BP // SAMPLE_BP), SAMPLE_BP, ann.n_tx, "shimmed reference oracle/_ref" if kind == "reference" else "oracle port", sys.version_info[0], sys.version_info[1])
    return bp / dt / 1e9, dt, kind, sample


def host_phases():
    """Host-side annotation parsing (outside every timed region): the product's read_gff and the reference's own on GTF text of
    the sample (the reference is ~1 ms per line, so it gets the first 2 000 lines only)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from magot_b200 import genome as mg_genome
    layout, contigs, ann = build_sample()
    gtf = ann.to_gtf([n for n, _ in layout])
    n_lines = gtf.count("\n")
    t0 = time.perf_counter()
    mg_genome.read_gff(gtf)
    t_prod = time.perf_counter() - t0
    out = {"gtf_lines": n_lines, "product_read_gff_lines_per_s": round(n_lines / t_prod)}
    try:
        import contextlib
        import io
        import ref_runner
        ref = ref_runner.ref()
        head = "\n".join(gtf.split("\n")[:2000]) + "\n"
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            ref.read_gff(head)
        out["reference_read_gff_lines_per_s"] = round(2000 / (time.perf_counter() - t0))
    except Exception as e:
        out["reference_read_gff_error"] = str(e)[:200]
    return out


def fasta_ingest_rates(device):
    """FASTA ingest (outside every timed region; SURVEY 8f-2): a 256 Mbp record with 60-column lines through
    mg_genome_pack_fasta (raw bytes to the device, line ends dropped there by K0f, packed by K0) next to what the host would
    spend only stripping the line ends (bytes.translate) and to the reference's own GenomeSequence loader (genome.py:856-877)
    on a 1/16 sample."""
    import numpy as np
    from magot_b200 import engine
    n = 256 << 20
    rng = np.random.default_rng(3)
    rows = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (n // 64, 61), dtype=np.uint8)]
    rows[:, 60] = 10
    raw = rows.reshape(-1)
    bases = (n // 64) * 60
    g = engine.DeviceGenome([bases], device=device)
    t0 = time.perf_counter()
    g.pack_fasta(0, raw)                                           # first pass: allocates the device buffers
    t_dev = time.perf_counter() - t0
    t0 = time.perf_counter()
    g.pack_fasta(0, raw)                                           # second pass: buffers exist, pages are warm
    t_dev2 = time.perf_counter() - t0
    g.finalize()
    assert g.fetch(0, bases - 120, bases) == raw[-122:].tobytes().translate(None, b"\n")
    g.close()
    data = raw.tobytes()
    t0 = time.perf_counter()
    data.translate(None, b"\r\n")
    t_host = time.perf_counter() - t0
    out = {"raw_bytes": int(raw.size), "pack_fasta_GBps_first": round(raw.size / t_dev / 1e9, 2),
           "pack_fasta_GBps": round(raw.size / t_dev2 / 1e9, 2), "host_strip_only_GBps": round(raw.size / t_host / 1e9, 2)}
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import ref_runner
        ref = ref_runner.ref()
        sample = ">c\n" + data[:raw.size // 16].decode("latin-1")
        t0 = time.perf_counter()
        ref.GenomeSequence(sample)
        out["reference_GenomeSequence_GBps"] = round(len(sample) / (time.perf_counter() - t0) / 1e9, 4)
    except Exception as e:
        out["reference_error"] = str(e)[:200]
    return out


def api_e2e(device):
    """Wall time of the PUBLIC API on config 3 at full size, from text to text (rank 0, outside every timed region):
    Genome(FASTA text) -> read_gff(GFF3 text) -> annotations.get_fasta('gene') for the CDS nucleotide product -- what
    genome_tools.gff2fasta does before it prints (genome_tools.py:324-330).  Split: FASTA ingest (header scan on the host, K0f + K0
    on the device), annotation parse (native reader), flatten (native, tops in Python-2.7 dict order), device + copy (K1-K2 and
    the text into a bytes object), decode (bytes -> the str the API returns)."""
    import numpy as np
    import torch
    from magot_b200 import engine, synth, genome as mg
    dev = torch.device("cuda", device)
    layout = synth.contig_layout("insect", 500_000_000, 3)
    parts = []
    for ci, (name, L) in enumerate(layout):              # the genome as 60-column FASTA text, produced on the device
        a = synth.synth_contig_device(L, 3 * 1000003 + ci * 64, dev).cpu().numpy()
        full = L // 60
        rows = np.empty((full, 61), dtype=np.uint8)
        rows[:, :60] = a[:full * 60].reshape(full, 60)
        rows[:, 60] = 10
        parts.append(b">" + name.encode() + b"\n" + rows.tobytes() + a[full * 60:].tobytes() + b"\n")
    fasta = b"".join(parts)
    del parts
    ann = synth.synth_annotation(layout, 60_000, 3)
    gff = ann.to_gff3([n for n, _ in layout])
    out = {"workload": "config 3 at full size through the public API: %.0f MB of FASTA text (500 Mbp, 2 000 scaffolds), %d lines of GFF3 text (30k genes / 60k mRNAs)" % (len(fasta) / 1e6, gff.count("\n"))}
    mg.TIMINGS = {}
    t0 = time.perf_counter()
    G = mg.Genome(fasta)
    t1 = time.perf_counter()
    G.read_gff(gff)
    t2 = time.perf_counter()
    text = G.annotations.get_fasta('gene')
    t3 = time.perf_counter()
    out.update({"fasta_ingest_s": round(t1 - t0, 3), "read_gff_s": round(t2 - t1, 3), "get_fasta_s": round(t3 - t2, 3),
                "total_s": round(t3 - t0, 3), "gff_lines_per_s": round(gff.count("\n") / (t2 - t1)),
                "fasta_GBps": round(len(fasta) / (t1 - t0) / 1e9, 2)})
    out.update({k: (round(v, 4) if isinstance(v, float) else v) for k, v in mg.TIMINGS.items()})
    out["spliced_Gbp_per_s_text_to_text"] = round(ann.spliced_bp("cds") / (t3 - t0) / 1e9, 4)
    out["spliced_Gbp_per_s_get_fasta_only"] = round(ann.spliced_bp("cds") / (t3 - t2) / 1e9, 4)
    assert text.count(">") == 60_000
    mg.TIMINGS = None
    G.genome_sequence.close()
    return out


def cpu_port_rate():
    """Single-threaded C restatement (oracle/oracle.c) on a larger sample: tight-loop CPU figure."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import coracle
    from magot_b200 import synth
    layout = synth.contig_layout("human", 60_000_000, SEED)
    contigs = synth.synth_genome_host(layout, SEED)
    ann = synth.synth_annotation(layout, 20_000, SEED)
    lens = np.array([a.size for a in contigs])
    raw = [a.tobytes() for a in contigs]
    t0 = time.perf_counter()
    bp = 0
    for which in ("cds", "exon"):
        tbl = ann.table(which, framing=False)
        lo = np.clip(tbl.seg_start - 1, 0, lens[tbl.seg_contig])
        hi = np.clip(tbl.seg_end, 0, lens[tbl.seg_contig])
        nuc, off = coracle.splice(raw, tbl.rec_seg_off, tbl.seg_contig, lo, hi, tbl.seg_strand)
        bp += nuc.size
        if which == "cds":
            coracle.splice_translate(nuc, off)
            bp += nuc.size
    dt = time.perf_counter() - t0
    return bp / dt / 1e9


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
def bind_to_gpu_cpus(local):
    """Pin this rank to the CPUs the GPU's PCIe root reports as local (NUMA placement of the pinned host buffers the
    device->host copies land in).  Returns what was done, for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bdf) as fh:
            txt = fh.read().strip()
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as fh:
            node = fh.read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                lo, hi = part.split("-")
                cpus.update(range(int(lo), int(hi) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"pci": bdf, "numa_node": node, "local_cpulist": txt, "bound_cpus": len(cpus)}
    except Exception as e:
        return {"error": str(e)[:120]}


class Workload(object):
    """One rank's batch: interval tables (host, pinned copies), device-resident plans and output buffers."""

    def __init__(self, g, ann, dev, streams):
        import numpy as np
        import torch
        from magot_b200 import _lib
        self.g, self.ann, self.dev, self.lib, self._lib = g, ann, dev, _lib.lib, _lib
        self.tables = {"cds": ann.table("cds"), "exon": ann.table("exon")}
        self.S_cds, self.S_exon = ann.spliced_bp("cds"), ann.spliced_bp("exon")
        self.bp_step = 2 * self.S_cds + self.S_exon
        self.stream, self.stream_b, self.stream_c = streams
        fields = ("rec_seg_off", "seg_contig", "seg_start", "seg_end", "seg_strand", "rec_lit_off", "rec_pre_len", "rec_suf_len", "lit")
        self.pinned = {k: {f: torch.from_numpy(np.array(getattr(t, f), copy=True)).pin_memory() for f in fields}
                       for k, t in self.tables.items()}
        self.h2d_bytes = sum(t.numel() * t.element_size() for k in self.pinned for t in self.pinned[k].values())
        self.plans = {k: self.create_plan(k, self.sp(self.stream)) for k in self.tables}
        self.sizes = {}
        for k in self.tables:
            a, b = ctypes.c_int64(0), ctypes.c_int64(0)
            _lib.check(self.lib.mg_plan_prepare(self.plans[k], _lib.MG_PROT_TRIMX, ctypes.byref(a), ctypes.byref(b), self.sp(self.stream)))
            self.sizes[k] = (a.value, b.value)
        # upper bounds of the text sizes from the HOST tables (sum of end-start+1 per segment + framing; a third of it for the
        # protein): with them K1 needs no host round trip (mg_plan_prepare_async) and K1 -> K2 -> K3 queue back to back
        self.caps = {}
        for k, t in self.tables.items():
            pay = t.approx_bytes_per_record() - t.rec_pre_len - t.rec_suf_len
            lit_bytes = int(t.rec_pre_len.astype(np.int64).sum() + t.rec_suf_len.astype(np.int64).sum())
            self.caps[k] = (int(pay.sum()) + lit_bytes, int((pay // 3).sum()) + lit_bytes)
            assert self.caps[k][0] >= self.sizes[k][0] and self.caps[k][1] >= self.sizes[k][1]
        pad = lambda n: (n + 31) // 32 * 32 + 32   # noqa: E731
        self.out = {"cds_n": torch.empty(pad(self.caps["cds"][0]), dtype=torch.uint8, device=dev),
                    "cds_p": torch.empty(pad(self.caps["cds"][1]), dtype=torch.uint8, device=dev),
                    "exon_n": torch.empty(pad(self.caps["exon"][0]), dtype=torch.uint8, device=dev)}
        self.d2h_bytes = self.sizes["cds"][0] + self.sizes["cds"][1] + self.sizes["exon"][0]
        self.last_heavy = None

    @staticmethod
    def sp(stream):
        return ctypes.c_void_p(stream.cuda_stream)

    @staticmethod
    def P(t):
        return ctypes.c_void_p(t.data_ptr())

    def create_plan(self, k, s):
        p, P = self.pinned[k], self.P
        h = ctypes.c_void_p()
        self._lib.check(self.lib.mg_plan_create(self.g.handle, self.tables[k].n_rec, P(p["rec_seg_off"]), self.tables[k].n_seg, P(p["seg_contig"]),
                                                P(p["seg_start"]), P(p["seg_end"]), P(p["seg_strand"]), P(p["rec_lit_off"]), P(p["rec_pre_len"]),
                                                P(p["rec_suf_len"]), P(p["lit"]), p["lit"].numel(), None, s, ctypes.byref(h)))
        return h

    def prepare_on(self, k, s, defer=False):
        """K1 without a host round trip.  defer: piece pass only (MG_PROT_DEFER); prepare_prot_on runs the record pass later."""
        flags = self._lib.MG_PROT_TRIMX | (self._lib.MG_PROT_DEFER if defer else 0)
        self._lib.check(self.lib.mg_plan_prepare_async(self.plans[k], flags, self.caps[k][0], self.caps[k][1], self.sp(s)))

    def prepare_prot_on(self, k, s):
        self._lib.check(self.lib.mg_plan_prepare_prot_async(self.plans[k], self.sp(s)))

    def step(self):
        """One pass of the hot path, device resident.  Three streams, nothing waits for the host: the CDS plan's K1 and K2 on
        `stream`, its K3 on `stream_c` (after K1), the exon plan's K1 and K2 on `stream_b`; kernels of different streams
        share the GPU (measured: 0.458 ms against 0.480 ms with the emit kernels put in series, scratch/overlap.py)."""
        import torch
        lib, chk, P = self.lib, self._lib.check, self.P
        mode = STEP_MODE
        if mode == "fused":
            # CDS plan: K1 -> K23 (nucleotide + protein text from one pass) on `stream`; exon plan: K1 -> K2 on `stream_b`
            self.prepare_on("cds", self.stream)
            chk(lib.mg_emit_nuc_prot_device(self.plans["cds"], P(self.out["cds_n"]), P(self.out["cds_p"]), self.sp(self.stream)))
            self.prepare_on("exon", self.stream_b)
            chk(lib.mg_emit_nuc_device(self.plans["exon"], P(self.out["exon_n"]), self.sp(self.stream_b)))
            return
        if mode == "multi":
            # both K1 side by side on two streams, then ONE launch for the three products (tiles interleaved for L2 reuse)
            self.prepare_on("exon", self.stream_b)
            self.prepare_on("cds", self.stream)
            self.stream.wait_stream(self.stream_b)
            chk(lib.mg_emit_products_device(self.plans["exon"], P(self.out["exon_n"]), self.plans["cds"], P(self.out["cds_n"]),
                                            P(self.out["cds_p"]), self.sp(self.stream)))
            return
        # K1 is two passes: pieces (what K2 needs) and records (amino-acid counts and protein offsets, what K3 needs).  The record
        # pass of the CDS plan runs on stream_c next to K2; the exon plan (nucleotide text only) never runs one.
        defer = STEP_DEFER
        self.prepare_on("cds", self.stream, defer=defer)
        e1 = torch.cuda.Event()
        e1.record(self.stream)
        chk(lib.mg_emit_nuc_device(self.plans["cds"], P(self.out["cds_n"]), self.sp(self.stream)))
        self.stream_c.wait_event(e1)
        if defer:
            self.prepare_prot_on("cds", self.stream_c)
        chk(lib.mg_emit_prot_device(self.plans["cds"], P(self.out["cds_p"]), self.sp(self.stream_c)))
        self.prepare_on("exon", self.stream_b, defer=defer)
        chk(lib.mg_emit_nuc_device(self.plans["exon"], P(self.out["exon_n"]), self.sp(self.stream_b)))

    def join(self):
        self.stream.wait_stream(self.stream_b)
        self.stream.wait_stream(self.stream_c)

    def capture(self, device):
        """The same step as a CUDA graph (mg_graph_begin/end): the exon plan forks to stream_b, the protein kernel to stream_c,
        both join `stream` again; one graph launch replays the 9 kernels + 2 memsets of the step."""
        import torch
        lib, chk, P, sp = self.lib, self._lib.check, self.P, self.sp
        self.step()                                      # everything a capture must not do (allocations) has happened
        self.join()
        torch.cuda.synchronize()
        s, sb, sc = sp(self.stream), sp(self.stream_b), sp(self.stream_c)
        chk(lib.mg_graph_begin(device, s))
        chk(lib.mg_stream_wait_stream(device, sb, s))
        self.prepare_on("exon", self.stream_b)
        chk(lib.mg_emit_nuc_device(self.plans["exon"], P(self.out["exon_n"]), sb))
        self.prepare_on("cds", self.stream)
        chk(lib.mg_stream_wait_stream(device, sc, s))
        chk(lib.mg_emit_nuc_device(self.plans["cds"], P(self.out["cds_n"]), s))
        chk(lib.mg_emit_prot_device(self.plans["cds"], P(self.out["cds_p"]), sc))
        chk(lib.mg_stream_wait_stream(device, s, sb))
        chk(lib.mg_stream_wait_stream(device, s, sc))
        g = ctypes.c_void_p()
        chk(lib.mg_graph_end(device, s, ctypes.byref(g)))
        self.graph = g
        return g

    def step_graph(self, device):
        self._lib.check(self.lib.mg_graph_launch(device, self.graph, self.sp(self.stream)))

    def kernel_times(self, reps):
        """Every kernel of the step alone on the GPU, in series on one stream with CUDA events around it (means of `reps`)."""
        import torch
        lib, chk, P = self.lib, self._lib.check, self.P
        ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731
        s, spp = self.stream, self.sp(self.stream)
        acc = {"k1_plan_cds_ms": 0.0, "k2_nuc_cds_ms": 0.0, "k3_prot_cds_ms": 0.0, "k1_plan_exon_ms": 0.0, "k2_nuc_exon_ms": 0.0}
        for _ in range(reps):
            e = [ev() for _ in range(6)]
            e[0].record(s)
            self.prepare_on("cds", s)                    # both passes of K1
            e[1].record(s)
            chk(lib.mg_emit_nuc_device(self.plans["cds"], P(self.out["cds_n"]), spp))
            e[2].record(s)
            chk(lib.mg_emit_prot_device(self.plans["cds"], P(self.out["cds_p"]), spp))
            e[3].record(s)
            self.prepare_on("exon", s, defer=STEP_DEFER)  # as in the step: piece pass only when the record pass is deferred
            e[4].record(s)
            chk(lib.mg_emit_nuc_device(self.plans["exon"], P(self.out["exon_n"]), spp))
            e[5].record(s)
            torch.cuda.synchronize()
            for i, k in enumerate(acc):
                acc[k] += e[i].elapsed_time(e[i + 1]) / reps
        return acc

    def fused_times(self, reps):
        """A/B of the fused forms (same bytes, tested bit-identical): K23 = mg_emit_nuc_prot_device (CDS nucleotide + protein text
        from one pass over the genome) and the one-launch emit of all three products (mg_emit_products_device, tiles interleaved
        for L2 reuse), each alone on the GPU with CUDA events around it."""
        import torch
        lib, chk, P = self.lib, self._lib.check, self.P
        s, spp = self.stream, self.sp(self.stream)
        self.prepare_on("cds", s)
        self.prepare_on("exon", s)
        acc = {"k23_nuc_prot_cds_ms": 0.0, "one_launch_three_products_ms": 0.0}
        for _ in range(reps):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            e[0].record(s)
            chk(lib.mg_emit_nuc_prot_device(self.plans["cds"], P(self.out["cds_n"]), P(self.out["cds_p"]), spp))
            e[1].record(s)
            e[2].record(s)
            chk(lib.mg_emit_products_device(self.plans["exon"], P(self.out["exon_n"]), self.plans["cds"], P(self.out["cds_n"]),
                                            P(self.out["cds_p"]), spp))
            e[3].record(s)
            torch.cuda.synchronize()
            acc["k23_nuc_prot_cds_ms"] += e[0].elapsed_time(e[1]) / reps
            acc["one_launch_three_products_ms"] += e[2].elapsed_time(e[3]) / reps
        return acc

    def check_totals(self):
        for k in self.tables:
            a, b = ctypes.c_int64(0), ctypes.c_int64(0)
            self._lib.check(self.lib.mg_plan_totals(self.plans[k], ctypes.byref(a), ctypes.byref(b), self.sp(self.stream)))
            want = tuple(self.sizes[k]) if not (STEP_DEFER and k == "exon") else (self.sizes[k][0], 0)   # exon plan: no record pass, no protein text
            assert (a.value, b.value) == want, (k, a.value, b.value, want)

    def close(self):
        for h in self.plans.values():
            self.lib.mg_plan_destroy(h)


STEP_MODE = os.environ.get("MAGOT_STEP", "streams3")     # streams3 | fused | multi  (see Workload.step)
STEP_DEFER = os.environ.get("MAGOT_STEP_DEFER", "1") != "0" and STEP_MODE == "streams3"   # record pass of K1 off the critical path
DUMP_SAMPLE = 4 << 20      # bytes kept per text over all ranks: 3 texts x 4 Mi x 4 B (float32) = 48 MiB in all


def dump_outputs(wl, out_dir, rank, world):
    """The three texts the last timed step left in HBM, as .npy files in out_dir, so that two builds can be compared output
    for output.  Each rank writes lengths<sfx>.npy (float64: bytes of its CDS nucleotide, CDS protein and exon transcript
    texts) and one float32 file per text with its bytes -- all of them when the text has at most DUMP_SAMPLE // world bytes,
    else the bytes at that many positions drawn with a fixed seed (ascending, repeats possible).  <sfx> is empty on one GPU
    and _rank<r> otherwise; the ranks split DUMP_SAMPLE, so a dump stays within 48 MiB whatever the number of GPUs."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    suffix = "_rank%d" % rank if world > 1 else ""
    cap = DUMP_SAMPLE // world
    texts = (("cds_nuc", "cds_n", wl.sizes["cds"][0]), ("cds_prot", "cds_p", wl.sizes["cds"][1]),
             ("exon_nuc", "exon_n", wl.sizes["exon"][0]))
    np.save(os.path.join(out_dir, "lengths%s.npy" % suffix), np.array([n for _, _, n in texts], dtype=np.float64))
    for name, key, n in texts:
        text = wl.out[key][:n]
        if n > cap:
            pos = np.sort(np.random.default_rng(SEED).integers(0, n, size=cap))
            text = text[torch.from_numpy(pos).to(text.device)]
        np.save(os.path.join(out_dir, "%s%s.npy" % (name, suffix)), text.cpu().numpy().astype(np.float32))


def profile_traffic():
    """DRAM bytes per launch of the emit kernels from the committed ncu capture (profiles/r2_traffic.json, written next to
    the .csv it was read from): not a literal in this file."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as fh:
            return json.load(fh)
    except Exception:
        return None


def gpu_arm(args):
    import numpy as np
    import torch
    from magot_b200 import _lib, engine, synth
    lib = _lib.lib
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.require_device(local)
    affinity = bind_to_gpu_cpus(local)
    stream = torch.cuda.Stream(device=dev)              # not the legacy default stream: that one cannot be captured in a CUDA graph
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)

    # ---- resident genome: synthesised on the device (torch, plumbing) and packed by K0
    t_setup = time.perf_counter()
    layout = synth.contig_layout("human", GENOME_BP, SEED)
    g = engine.DeviceGenome([l for _, l in layout], device=local)
    t_pack = 0.0
    CH = 256 << 20
    for ci, (_, L) in enumerate(layout):
        for off in range(0, L, CH):
            n = min(CH, L - off)
            a = synth.synth_contig_device(n, SEED * 1000003 + ci * 64 + off // CH, dev)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            g.pack_device(ci, a.data_ptr(), n, offset=off, stream=sp)
            torch.cuda.synchronize()
            t_pack += time.perf_counter() - t0
            del a
    g.finalize()
    torch.cuda.empty_cache()

    # ---- the batch of config 4: 200k transcripts, the SAME on every rank (strong scaling): rank k takes the k-th of `world`
    # contiguous shards of ~equal output bytes (engine.shard_bounds), texts are gathered in record order on the host
    ann_all = synth.synth_annotation(layout, N_TX, SEED)
    cds_bp = np.add.reduceat(ann_all.cds_end - ann_all.cds_start + 1, ann_all.cds_off[:-1]) if ann_all.cds_off[-1] else np.zeros(ann_all.n_tx)
    cds_bp = np.where(np.diff(ann_all.cds_off) > 0, cds_bp, 0)
    exon_bp = np.add.reduceat(ann_all.exon_end - ann_all.exon_start + 1, ann_all.exon_off[:-1])
    weights = cds_bp * (4.0 / 3.0) + exon_bp + 3 * 12
    bounds = engine.shard_bounds(weights, world)
    ann = ann_all.subset(np.arange(bounds[rank], bounds[rank + 1])) if world > 1 else ann_all
    streams = (stream, torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev))
    wl = Workload(g, ann, dev, streams)
    setup_s = time.perf_counter() - t_setup
    ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    use_graph = os.environ.get("MAGOT_BENCH_GRAPH", "0") != "0"   # measured: eager 0.4606 / graph 0.4635 ms at N=1, 0.0851 / 0.0948 ms per step at N=8
    # (successive eager steps overlap on the three streams, a graph replay starts only when the previous one has drained)

    def timed_loop(w, warmup, steps):
        """K timed steps; with use_graph each step is one replay of the captured step (same kernels, same streams)."""
        l0 = lib.mg_kernel_launches()
        w.step()
        w.join()
        per_step = lib.mg_kernel_launches() - l0         # kernels of one step, counted on an eager step
        if use_graph:
            w.capture(local)
            run = lambda: w.step_graph(local)            # noqa: E731
        else:
            run = w.step
        for _ in range(warmup):
            run()
        w.join()
        barrier()
        s_ev, e_ev = ev(), ev()
        s_ev.record(stream)
        for _ in range(steps):
            run()
        w.join()
        e_ev.record(stream)
        barrier()
        if use_graph:
            lib.mg_graph_destroy(w.graph)
        return s_ev.elapsed_time(e_ev) / steps, per_step * steps

    clocks = ClockSampler(local)
    clocks.start()
    dev_ms, launches = timed_loop(wl, args.warmup, args.steps)
    wl.check_totals()
    if args.dump_outputs:
        dump_outputs(wl, args.dump_outputs, rank, world)
    kt = wl.kernel_times(max(3, min(args.steps, 10)))
    ft = wl.fused_times(max(3, min(args.steps, 10))) if world == 1 else None

    # ---- weak-scaling supplement (N > 1): every rank its own 200k-transcript batch, nothing shared
    weak = None
    if world > 1:
        wl_w = Workload(g, synth.synth_annotation(layout, N_TX, SEED + 1000 * rank), dev, streams)
        w_ms, _ = timed_loop(wl_w, args.warmup, args.steps)
        t = torch.tensor([w_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        bpw = torch.tensor([float(wl_w.bp_step)], dtype=torch.float64, device=dev)
        dist.all_reduce(bpw, op=dist.ReduceOp.SUM)
        weak = {"value": float(bpw.item()) / (float(t.item()) * 1e-3) / 1e9, "unit": "Gbp/s", "ms_per_step": float(t.item()),
                "note": "every rank runs its own %d-transcript batch over the replicated genome (no shared work)" % N_TX}
        wl_w.close()
        del wl_w
        torch.cuda.empty_cache()

    # ---- end to end through the C ABI with HOST buffers, texts gathered in record order in ONE host buffer per product.
    # N > 1: the three final texts live in POSIX shared memory (/dev/shm) mapped by every rank; a rank page-locks the slice its
    # shard owns (cudaHostRegister) and copies its texts straight to their final place over its own PCIe link: the "final host
    # gather" of north_star without a second copy and without NCCL.  Successive steps are double-buffered (two stream pairs,
    # two host buffer sets), the way a caller streaming batches would do it: the device->host copies of step i overlap the
    # table upload and the kernels of step i+1.  Every step uploads its own interval tables from pinned host memory.
    sizes3 = [wl.sizes["cds"][0], wl.sizes["cds"][1], wl.sizes["exon"][0]]
    if dist is not None:
        allsz = torch.zeros((world, 3), dtype=torch.int64, device=dev)
        allsz[rank] = torch.tensor(sizes3, dtype=torch.int64, device=dev)
        dist.all_reduce(allsz, op=dist.ReduceOp.SUM)
        allsz = allsz.cpu().numpy()
    else:
        allsz = np.array([sizes3], dtype=np.int64)
    offs = np.concatenate((np.zeros((1, 3), dtype=np.int64), np.cumsum(allsz, axis=0)))      # [world+1, 3]
    totals3 = offs[-1]
    host_sets, shm_paths, registered = [], [], []
    cudart = torch.cuda.cudart()
    for si in range(2):
        bufs = []
        for j in range(3):
            n = int(totals3[j])
            if dist is None:
                bufs.append(torch.empty(max(n, 1), dtype=torch.uint8, pin_memory=True))
                continue
            path = "/dev/shm/magot_bench_%s_%d_%d" % (os.environ.get("MASTER_PORT", "0"), si, j)
            if rank == 0:
                with open(path, "wb") as fh:
                    fh.truncate(max(n, 1))
                shm_paths.append(path)
            dist.barrier()
            t = torch.from_file(path, shared=True, size=max(n, 1), dtype=torch.uint8)
            lo, hi = int(offs[rank][j]), int(offs[rank + 1][j])
            if hi > lo:                                  # page-lock this rank's slice (page-aligned superset)
                a0 = (t.data_ptr() + lo) // 4096 * 4096
                a1 = -(-(t.data_ptr() + hi) // 4096) * 4096
                a1 = min(a1, t.data_ptr() + -(-max(n, 1) // 4096) * 4096)
                rc = cudart.cudaHostRegister(a0, a1 - a0, 0)
                assert int(rc) == 0, "cudaHostRegister failed: %s" % rc
                registered.append(a0)
            bufs.append(t)
        host_sets.append(bufs)
    pairs = [(stream, streams[1]), (torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev))]
    in_flight = [None, None]
    my_off = [int(x) for x in offs[rank]]

    def HP(t, off):
        return ctypes.c_void_p(t.data_ptr() + off)

    def e2e_retire(slot):
        if in_flight[slot] is not None:
            hc, he, sa, sb = in_flight[slot]
            _lib.check(lib.mg_stream_sync(local, sa))
            _lib.check(lib.mg_stream_sync(local, sb))
            lib.mg_plan_destroy(hc)
            lib.mg_plan_destroy(he)
            in_flight[slot] = None

    def e2e_step(i):
        slot = i & 1
        e2e_retire(slot)
        sa = ctypes.c_void_p(pairs[slot][0].cuda_stream)
        sb = ctypes.c_void_p(pairs[slot][1].cuda_stream)
        hs = host_sets[slot]
        hc = wl.create_plan("cds", sa)
        he = wl.create_plan("exon", sb)
        a, b = ctypes.c_int64(0), ctypes.c_int64(0)
        _lib.check(lib.mg_plan_prepare(hc, _lib.MG_PROT_TRIMX, ctypes.byref(a), ctypes.byref(b), sa))
        _lib.check(lib.mg_emit_nuc_host(hc, HP(hs[0], my_off[0]), sa))
        _lib.check(lib.mg_emit_prot_host(hc, HP(hs[1], my_off[1]), sa))
        _lib.check(lib.mg_plan_prepare(he, _lib.MG_PROT_TRIMX, ctypes.byref(a), ctypes.byref(b), sb))
        _lib.check(lib.mg_emit_nuc_host(he, HP(hs[2], my_off[2]), sb))
        in_flight[slot] = (hc, he, sa, sb)

    for i in range(max(2, min(args.warmup, 4))):
        e2e_step(i)
    e2e_retire(0)
    e2e_retire(1)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(i)
    e2e_retire(0)
    e2e_retire(1)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps      # host clock around fully synchronised work on four streams
    barrier()
    # this rank's slices hold what the device-resident step produced, at their place in the gathered texts
    for hs in host_sets:
        for j, key in enumerate(("cds_n", "cds_p", "exon_n")):
            n = sizes3[j]
            assert torch.equal(hs[j][my_off[j]:my_off[j] + n], wl.out[key][:n].cpu()), "end-to-end text differs from the device-resident text"
    gather_check = None
    if dist is not None:
        dist.barrier()
        if rank == 0:                                    # record order across the shards: shard k starts with its first transcript's header
            ok = True
            for k in range(world):
                if bounds[k + 1] > bounds[k]:
                    want = (">" + ann_all.names[bounds[k]] + "\n").encode()
                    for j in (0, 1, 2):
                        o = int(offs[k][j])
                        ok = ok and bytes(host_sets[0][j][o:o + len(want)].numpy().tobytes()) == want
            gather_check = bool(ok)
            assert ok, "gathered texts are not in record order"

    # ---- bare device->host ceiling of this box: every rank copies as many bytes as its step moves, nothing else running
    probe_src = torch.empty(max(wl.d2h_bytes, 1), dtype=torch.uint8, device=dev)
    reps = 4
    def d2h_probe():
        o = 0
        for j in range(3):
            n = sizes3[j]
            if n:
                _lib.check(lib.mg_copy_d2h_async(local, HP(host_sets[0][j], my_off[j]), ctypes.c_void_p(probe_src.data_ptr() + o), n, sp))
            o += n
    d2h_probe()
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        d2h_probe()
    torch.cuda.synchronize()
    probe_ms = (time.perf_counter() - t0) * 1e3 / reps
    barrier()
    del probe_src
    clk = clocks.stop()
    for a0 in registered:
        cudart.cudaHostUnregister(a0)
    del host_sets
    if dist is not None:
        dist.barrier()
        if rank == 0:
            for pth in shm_paths:
                try:
                    os.unlink(pth)
                except OSError:
                    pass

    # ---- config 5 (extra information, outside the timed steps): six-frame ORF scan of the whole genome, min ORF 100 aa
    six = None
    if not args.no_sixframe:
        try:
            # contigs are independent: each rank scans its LPT share of the contigs (longest first, each to the least loaded
            # GPU; strong scaling, no exchange step); time = max over ranks, ORFs and residues summed
            from magot_b200 import orfs as _orfs
            shard = _orfs.lpt_shards([l for _, l in layout], world)[rank]
            ids = np.ascontiguousarray(shard, dtype=np.int64)
            my_bp = sum(layout[c][1] for c in shard)
            n_orf, n_bytes = ctypes.c_int64(0), ctypes.c_int64(0)

            def six_count():
                _lib.check(lib.mg_sixframe_count_list(g.handle, ids.size, ctypes.c_void_p(ids.ctypes.data), 100, ctypes.byref(n_orf),
                                                      ctypes.byref(n_bytes), sp))
            torch.cuda.synchronize()
            f0, f1 = ev(), ev()
            f0.record(stream)
            six_count()                                  # first call on this genome: builds the stop-codon index (2 bits/base), then scans
            f1.record(stream)
            torch.cuda.synchronize()
            t_first = f0.elapsed_time(f1)
            aa_dev = torch.empty((n_bytes.value + 31) // 32 * 32 + 32, dtype=torch.uint8, device=dev)
            scans, emits = [], []
            for _ in range(5):
                a0, a1, a1b, a2 = ev(), ev(), ev(), ev()
                a0.record(stream)
                six_count()
                a1.record(stream)
                a1b.record(stream)
                _lib.check(lib.mg_sixframe_emit_device(g.handle, ctypes.c_void_p(aa_dev.data_ptr()), None, sp))
                a2.record(stream)
                torch.cuda.synchronize()
                scans.append(a0.elapsed_time(a1))
                emits.append(a1b.elapsed_time(a2))
            t_scan, t_emit = sorted(scans)[2], sorted(emits)[2]
            tot_orf, tot_bytes, max_bp = n_orf.value, n_bytes.value, my_bp
            if dist is not None:
                tt = torch.tensor([t_scan, t_emit, float(my_bp), t_first], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                t_scan, t_emit, max_bp, t_first = [float(x) for x in tt.tolist()]
                ts = torch.tensor([n_orf.value, n_bytes.value], dtype=torch.float64, device=dev)
                dist.all_reduce(ts, op=dist.ReduceOp.SUM)
                tot_orf, tot_bytes = [int(x) for x in ts.tolist()]
            six = {"workload": "config 5: six-frame translation + ORF scan of the whole genome, min ORF 100 aa (reference semantics of Sequence.get_orfs)",
                   "sharding": "contigs assigned to %d GPU(s) longest-first to the least loaded (LPT); largest share %.3f Gbp; strong scaling, "
                               "times are the max over ranks" % (world, max_bp / 1e9),
                   "orfs": tot_orf, "aa_bytes": tot_bytes, "scan_ms": round(t_scan, 3), "emit_ms": round(t_emit, 3),
                   "first_scan_ms_incl_index_build": round(t_first, 3),
                   "timing": "median of 5 calls (mg_sixframe_count_list incl. its host round trip for the ORF count, then mg_sixframe_emit_device), CUDA events; "
                             "the first call on a genome also builds the stop-codon index (0.25 B/base, like the reverse plane a property of the packed genome) and is reported apart",
                   "genome_Gbp_per_s": round(GENOME_BP / ((t_scan + t_emit) * 1e-3) / 1e9, 1),
                   "six_frame_Gbp_per_s": round(6 * GENOME_BP / ((t_scan + t_emit) * 1e-3) / 1e9, 1),
                   "algorithmic_GBps": round((GENOME_BP * 0.5 + tot_bytes + 32 * tot_orf) / ((t_scan + t_emit) * 1e-3) / 1e9, 1),
                   "genome_Gbp_per_s_first_call": round(GENOME_BP / ((t_first + t_emit) * 1e-3) / 1e9, 1),
                   "bound": "scan: latency of the per-tile / per-row prologues (0.78 GB of index read in ~0.2 ms); residues: instruction issue (k_six_aa); see DESIGN.md section 4"}
            del aa_dev
        except Exception as e:
            six = {"error": str(e)[:300]}
            if dist is not None:
                raise

    # ---- max over ranks (times), sums over ranks (work)
    kt_keys = list(kt)
    if dist is not None:
        t = torch.tensor([dev_ms, e2e_ms, probe_ms] + [kt[k] for k in kt_keys], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        vals = [float(x) for x in t.tolist()]
        dev_ms, e2e_ms, probe_ms = vals[:3]
        kt_max = dict(zip(kt_keys, vals[3:]))
        tot = torch.tensor([wl.bp_step, wl.h2d_bytes, wl.d2h_bytes, launches], dtype=torch.float64, device=dev)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        bp_all, h2d_all, d2h_all, launches_all = [float(x) for x in tot.tolist()]
    else:
        kt_max = dict(kt)
        bp_all, h2d_all, d2h_all, launches_all = wl.bp_step, wl.h2d_bytes, wl.d2h_bytes, launches

    # ---- roofline (this rank's shard; at N = 1 the whole batch).  Algorithmic bytes per SURVEY 8d:
    #   K2: S*0.5 (packed read) + text written + 14 B/segment + 8 B/record (+ literal bytes read)
    #   K3: S*0.5 + protein text written + 14 B/segment + 16 B/record
    #   K1: 14 B/segment + 8 B/record read, 16 B/piece + 16 B/record of derived tables written
    peak, peak_src = peaks()
    T = wl.tables

    def alg_k2(S, tbl, text):
        return S * 0.5 + text + tbl.n_seg * 14 + tbl.n_rec * 8 + tbl.lit.size

    ab_cds, ab_exon = alg_k2(wl.S_cds, T["cds"], wl.sizes["cds"][0]), alg_k2(wl.S_exon, T["exon"], wl.sizes["exon"][0])
    ab_k3 = wl.S_cds * 0.5 + wl.sizes["cds"][1] + T["cds"].n_seg * 14 + T["cds"].n_rec * 16
    ab_k1 = {k: T[k].n_seg * 14 + T[k].n_rec * 8 + (T[k].n_seg + 2 * T[k].n_rec) * 16 + T[k].n_rec * 16 for k in T}
    k2_ms = kt["k2_nuc_cds_ms"] + kt["k2_nuc_exon_ms"]
    ach = (ab_cds + ab_exon) / (k2_ms * 1e-3) / 1e9
    step_alg = ab_cds + ab_exon + ab_k3 + ab_k1["cds"] + ab_k1["exon"]
    gbps = lambda b, ms: round(b / ms / 1e6, 1) if ms > 0 else None   # noqa: E731
    traffic = profile_traffic()
    roofline = {"kernel": "k_emit_nuc (K2 splice + per-segment RC + FASTA framing)", "bound": "hbm", "achieved": round(ach, 1),
                "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                "traffic": (traffic or {}).get("k_emit_nuc_mean_bytes_per_launch") if (GENOME_BP == 3_100_000_000 and N_TX == 200_000 and world == 1) else None,
                "traffic_source": (traffic or {}).get("source"),
                "peak_source": peak_src, "frac_of_nominal_8TBs": round(ach / 8000.0, 4),
                "launches_per_step": 2, "avg_launch_ms": round(k2_ms / 2, 4), "algorithmic_bytes_per_launch": int((ab_cds + ab_exon) / 2),
                "timing": "each kernel alone on the GPU, in series on one stream, CUDA events around it, mean of %d passes after the timed steps" % max(3, min(args.steps, 10)),
                "per_kernel": {
                    "k2_nuc_cds": {"ms": round(kt["k2_nuc_cds_ms"], 4), "alg_bytes": int(ab_cds), "GBps": gbps(ab_cds, kt["k2_nuc_cds_ms"]), "frac": round(ab_cds / kt["k2_nuc_cds_ms"] / 1e6 / peak, 4)},
                    "k2_nuc_exon": {"ms": round(kt["k2_nuc_exon_ms"], 4), "alg_bytes": int(ab_exon), "GBps": gbps(ab_exon, kt["k2_nuc_exon_ms"]), "frac": round(ab_exon / kt["k2_nuc_exon_ms"] / 1e6 / peak, 4)},
                    "k3_prot_cds": {"ms": round(kt["k3_prot_cds_ms"], 4), "alg_bytes": int(ab_k3), "GBps": gbps(ab_k3, kt["k3_prot_cds_ms"]), "frac": round(ab_k3 / kt["k3_prot_cds_ms"] / 1e6 / peak, 4)},
                    "k1_plan_cds": {"ms": round(kt["k1_plan_cds_ms"], 4), "alg_bytes": int(ab_k1["cds"]), "GBps": gbps(ab_k1["cds"], kt["k1_plan_cds_ms"]), "frac": round(ab_k1["cds"] / kt["k1_plan_cds_ms"] / 1e6 / peak, 4)},
                    "k1_plan_exon": {"ms": round(kt["k1_plan_exon_ms"], 4), "alg_bytes": int(ab_k1["exon"]), "GBps": gbps(ab_k1["exon"], kt["k1_plan_exon_ms"]), "frac": round(ab_k1["exon"] / kt["k1_plan_exon_ms"] / 1e6 / peak, 4)}},
                "fused_ab": None if ft is None else {
                    "k23_nuc_prot_cds": {"ms": round(ft["k23_nuc_prot_cds_ms"], 4), "vs_k2_plus_k3_ms": round(kt["k2_nuc_cds_ms"] + kt["k3_prot_cds_ms"], 4),
                                         "alg_bytes": int(ab_cds + wl.sizes["cds"][1]), "frac": round((ab_cds + wl.sizes["cds"][1]) / ft["k23_nuc_prot_cds_ms"] / 1e6 / peak, 4),
                                         "dram_read_MB": ((traffic or {}).get("k23") or {}).get("dram_read_MB"), "k2_plus_k3_dram_read_MB": ((traffic or {}).get("k23") or {}).get("k2_plus_k3_dram_read_MB")},
                    "one_launch_three_products": {"ms": round(ft["one_launch_three_products_ms"], 4),
                                                  "vs_three_launches_ms": round(kt["k2_nuc_cds_ms"] + kt["k3_prot_cds_ms"] + kt["k2_nuc_exon_ms"], 4),
                                                  "dram_read_MB": ((traffic or {}).get("multi") or {}).get("dram_read_MB"),
                                                  "three_launches_dram_read_MB": ((traffic or {}).get("multi") or {}).get("three_launches_dram_read_MB")},
                    "note": "both fused forms cut the DRAM reads of a step (ncu, profiles/) but not its time: the emit kernels are bound by issue slots and L1 wavefronts, "
                            "not by DRAM; the timed step therefore keeps K2 / K3 / K2 on three streams (MAGOT_STEP=fused|multi select the fused forms)"},
                "step_alg_bytes": int(step_alg), "step_frac": round(step_alg / (dev_ms * 1e-3) / 1e9 / peak, 4),
                "step_note": "step_frac = algorithmic bytes of all kernels of this rank's step / the step time (kernels of the three streams overlap) / peak",
                "sum_of_kernels_alone_ms": round(sum(kt.values()), 4)}

    line = None
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                v, dt, kind, sample = cpu_reference_rate(1, 0, 1)
                cpu = {"value": v, "unit": "Gbp/s", "cores": 1, "kind": kind, "sample": sample, "seconds": round(dt, 2),
                       "host_cpus": os.cpu_count()}
                try:
                    cpu["c_port_single_thread_Gbps"] = round(cpu_port_rate(), 4)
                except Exception as e:      # the C port is extra information only
                    cpu["c_port_error"] = str(e)[:200]
                try:
                    cpu["host_annotation_parse"] = host_phases()
                except Exception as e:
                    cpu["host_annotation_parse"] = {"error": str(e)[:200]}
                try:
                    cpu["api_e2e"] = api_e2e(local)
                except Exception as e:
                    cpu["api_e2e"] = {"error": str(e)[:300]}
                try:
                    cpu["fasta_ingest"] = fasta_ingest_rates(local)
                except Exception as e:
                    cpu["fasta_ingest"] = {"error": str(e)[:200]}
            except Exception as e:
                cpu = {"value": None, "unit": "Gbp/s", "cores": 1, "kind": "port", "sample": "failed: %s" % str(e)[:300]}
        value = bp_all / (dev_ms * 1e-3) / 1e9
        e2e_v = bp_all / (e2e_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": "config 4: synthetic %.2f Gbp human-scale genome (replicated per GPU; forward + reverse-complement planes, 0.5 B/base each) + ONE %d-transcript GTF-shaped batch cut into %d contiguous byte-balanced shard(s), one per GPU (strong scaling); products: CDS nucleotide FASTA + CDS protein FASTA + exon-based transcript FASTA; e2e gathers the three texts in record order in one host buffer each" % (GENOME_BP / 1e9, N_TX, world),
                       "genome_bp": GENOME_BP, "transcripts": N_TX, "transcripts_this_rank": int(ann.n_tx), "cds_segments_this_rank": int(T["cds"].n_seg),
                       "exons_this_rank": int(T["exon"].n_seg), "spliced_cds_bp_this_rank": wl.S_cds, "spliced_exon_bp_this_rank": wl.S_exon,
                       "bp_per_step_all_ranks": int(bp_all),
                       "parallelism": "transcript shards per GPU, genome replicated, no collective on the data path (NCCL only for barriers and the max/sum of timing scalars); per GPU three CUDA streams: CDS piece pass -> K2 | CDS record pass -> K3 | exon piece pass -> K2 (K1's record pass is deferred off the critical path, MG_PROT_DEFER)",
                       "l2": "no flush: each step streams ~%.2f GB of distinct output + genome lines per GPU, far above the 126 MB L2" % ((wl.d2h_bytes + 0.5 * wl.bp_step) / 1e9),
                       "genome_device_bytes": int(g.device_bytes()), "pack_s": round(t_pack, 3), "setup_s": round(setup_s, 1),
                       "cpu_affinity": affinity},
            "clocks": clk,
            "e2e": {"value": e2e_v, "unit": "Gbp/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all),
                    "d2h_achieved_GBps": round(d2h_all / (e2e_ms * 1e-3) / 1e9, 2),
                    "d2h_roof_GBps": round(d2h_all / (probe_ms * 1e-3) / 1e9, 2),
                    "d2h_roof_note": "bare probe on the same box and buffers: every rank copies its step's %d-byte share device->host with nothing else running, max over ranks" % int(wl.d2h_bytes),
                    "gather": ("texts of the %d shards land in one POSIX-shared-memory buffer per product (each rank page-locks and fills its own slice); record order checked: %s" % (world, gather_check)) if world > 1 else "single GPU: one pinned buffer per product"},
            "gpu_launches": int(launches_all),
            "roofline": roofline,
        }
        if weak is not None:
            line["weak"] = weak
        if six is not None:
            line["sixframe"] = six
        if cpu is not None:
            line["cpu_baseline"] = cpu
    wl.close()
    g.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line))


def reference_arm(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    workers = max(1, min(os.cpu_count() or 1, 32))
    warm = max(0, args.warmup)
    v, dt, kind, sample = cpu_reference_rate(max(args.steps, 1), warm, workers)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Gbp/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": "config 4, BOUNDED SAMPLE (not the full batch): the config-4 generators at 1/%d scale (%d bp genome, %d transcripts); "
                                   "each step = the reference's own get_fasta over the sample for the three products (CDS nucleotide, CDS protein, "
                                   "exon transcripts) on %d host processes (the reference is single-threaded; a multiprocessing pool over genes is the "
                                   "most it can use); the reference's objects are built directly, its read_gff (~1 ms per line) is EXCLUDED from the "
                                   "timed region; rate in Gbp/s, so the ratio to the GPU arm is a rate ratio, not a same-input ratio"
                                   % (max(1, GENOME_BP // SAMPLE_BP), SAMPLE_BP, SAMPLE_TX, workers),
                       "sample_genome_bp": SAMPLE_BP, "sample_transcripts": SAMPLE_TX, "host_processes": workers, "host_cpus": os.cpu_count()},
            "cpu_baseline": {"value": v, "unit": "Gbp/s", "cores": workers, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="magot_b200", choices=["magot_b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sixframe", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the texts of the last timed step to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path only")
    if args.impl == "reference":
        reference_arm(args)
    else:
        args.warmup = max(args.warmup, 3)
        gpu_arm(args)


if __name__ == "__main__":
    main()
