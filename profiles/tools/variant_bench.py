"""Variant consequences on config 4's genome and CDS plan: 4 M SNVs and 0.5 M indels of 1 to 10 bases drawn over the whole
genome, and 0.2 M SNVs placed inside CDS payloads, REF read from the genome (seeded).  Times mg_plan_variant_count (upload,
status and normalisation, join, scan, merge; it returns a row count, so it ends in a synchronise: host clock and CUDA events)
and mg_plan_variant_emit_device (CUDA events), medians over REPS calls after WARM warm-up calls, then a torch.profiler run of
one count + emit for the per-kernel split and the host-to-device copies.  The genome and the table come from the seeds and
generators k1_bench.py uses.  Prints one JSON line with the card's name, power limit and SM clock read in the same run.

    python profiles/tools/variant_bench.py [tag]        env: VRB_REPS (default 20), VRB_WARM (3), MAGOT_BENCH_TX (200000)
"""
import ctypes
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))   # repo root
import numpy as np
import torch

from magot_b200 import _lib, engine, synth
import k1_bench

lib = _lib.lib
REPS = int(os.environ.get("VRB_REPS", 20))
WARM = int(os.environ.get("VRB_WARM", 3))
N_SNV, N_INDEL, N_CDS_SNV = 4_000_000, 500_000, 200_000


def alleles(rng, lens, contig_dev, tbl):
    """(contig, pos, allele_off, bytes) of the seeded allele set, sorted by (contig, pos)."""
    total = int(lens.sum())
    cum = np.concatenate(([0], np.cumsum(lens)))
    g = rng.integers(0, total, size=N_SNV + N_INDEL)
    contig = np.searchsorted(cum, g, side="right") - 1
    pos = g - cum[contig]
    # CDS SNVs: a random CDS segment, a random base of it (segments are 1-based inclusive on the forward strand)
    e = rng.integers(0, tbl.n_seg, size=N_CDS_SNV)
    c2 = tbl.seg_contig[e].astype(np.int64)
    lo = np.clip(tbl.seg_start[e] - 1, 0, lens[c2])
    hi = np.clip(tbl.seg_end[e], 0, lens[c2])
    ok = hi > lo
    c2, p2 = c2[ok], lo[ok] + (rng.random(int(ok.sum())) * (hi[ok] - lo[ok])).astype(np.int64)
    contig, pos = np.concatenate((contig, c2)), np.concatenate((pos, p2))
    n = contig.size
    kind = np.zeros(n, np.int8)                               # 0 SNV, 1 insertion, 2 deletion
    kind[N_SNV:N_SNV + N_INDEL] = 1 + (rng.random(N_INDEL) < 0.5)
    k = rng.integers(1, 11, size=n)
    ref_len = np.where(kind == 2, k + 1, 1)
    pos = np.minimum(pos, lens[contig] - ref_len)
    order = np.lexsort((pos, contig))
    contig, pos, kind, k, ref_len = contig[order], pos[order], kind[order], k[order], ref_len[order]
    win = np.zeros((n, 11), np.uint8)                         # REF bytes from the device copy of each contig
    for c in range(len(lens)):
        sel = np.flatnonzero(contig == c)
        if sel.size:
            idx = torch.from_numpy(pos[sel]).to(contig_dev[c].device)[:, None] + torch.arange(11, device=contig_dev[c].device)
            win[sel] = contig_dev[c][idx.clamp_(max=int(lens[c]) - 1)].cpu().numpy()
    bases = np.frombuffer(b"ACGT", np.uint8)
    up = win[:, 0] & 0xDF
    alt_snv = bases[(np.searchsorted(bases, np.where(np.isin(up, bases), up, 65)) + rng.integers(1, 4, size=n)) % 4]
    ins = bases[rng.integers(0, 4, size=(n, 10))]
    parts, lens_out = [], np.zeros(2 * n, np.int64)
    for i in range(n):
        r = win[i, :ref_len[i]].tobytes()
        if kind[i] == 0:
            a = bytes([alt_snv[i]])
        elif kind[i] == 1:
            a = r + ins[i, :k[i]].tobytes()
        else:
            a = r[:1]
        parts.append(r)
        parts.append(a)
        lens_out[2 * i], lens_out[2 * i + 1] = len(r), len(a)
    off = np.concatenate(([0], np.cumsum(lens_out))).astype(np.int64)
    return contig.astype(np.int32), pos.astype(np.int64), off, b"".join(parts)


def main():
    tag = sys.argv[1] if len(sys.argv) > 1 else ""
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)
    layout = synth.contig_layout("human", k1_bench.GENOME_BP, k1_bench.SEED)
    lens = np.array([n for _, n in layout], dtype=np.int64)
    g = engine.DeviceGenome(lens, device=0)
    CH = 256 << 20
    contig_dev = []
    for ci, (_, L) in enumerate(layout):
        whole = torch.empty(L, dtype=torch.uint8, device=dev)
        for off in range(0, L, CH):
            n = min(CH, L - off)
            a = synth.synth_contig_device(n, k1_bench.SEED * 1000003 + ci * 64 + off // CH, dev)
            g.pack_device(ci, a.data_ptr(), n, offset=off, stream=sp)
            torch.cuda.synchronize()
            whole[off:off + n] = a
            del a
        contig_dev.append(whole)
    g.finalize()
    t = synth.synth_annotation(layout, k1_bench.N_TX, k1_bench.SEED).table("cds")
    contig, pos, off, buf = alleles(np.random.default_rng(k1_bench.SEED), lens, contig_dev, t)
    del contig_dev
    torch.cuda.empty_cache()
    plan = engine.Plan(g, t, stream=sp)
    plan.prepare_async(trimx=False, defer_records=True)
    torch.cuda.synchronize()
    n_var = contig.size
    status = np.zeros(n_var, np.int8)
    n_rows = ctypes.c_int64(0)
    P = lambda a: ctypes.c_void_p(a.ctypes.data)   # noqa: E731

    def count():
        _lib.check(lib.mg_plan_variant_count(plan.handle, n_var, P(contig), P(pos), P(off), buf, len(buf), 0, None, P(status),
                                             ctypes.byref(n_rows), sp))

    count()
    d_rows = torch.empty(max(1, n_rows.value) * 64, dtype=torch.uint8, device=dev)
    emit = lambda: _lib.check(lib.mg_plan_variant_emit_device(plan.handle, ctypes.c_void_p(d_rows.data_ptr()), sp))   # noqa: E731
    res = {"tag": tag, "card": k1_bench.card(), "reps": REPS, "n_tx": k1_bench.N_TX, "n_rec": int(t.n_rec), "n_seg": int(t.n_seg),
           "n_alleles": int(n_var), "allele_bytes": len(buf)}
    for _ in range(WARM):
        count()
    host, evs = [], []
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record(stream)
        count()
        b.record(stream)
        host.append((time.perf_counter() - t0) * 1e3)
        evs.append((a, b))
    torch.cuda.synchronize()
    res["count_host_ms_med"] = round(float(np.median(host)), 3)
    res["count_events_ms_med"] = round(float(np.median([a.elapsed_time(b) for a, b in evs])), 3)
    k1_bench.REPS, k1_bench.WARM = max(REPS, 50), WARM
    res["emit"] = k1_bench.timed(emit, stream)
    res["rows"] = int(n_rows.value)
    res["status_counts"] = np.bincount(status.astype(np.int64), minlength=4).tolist()
    rows = d_rows.cpu().numpy()[:n_rows.value * 64].view(engine.VEF_DTYPE)
    res["class_counts"] = dict(zip(_lib.VEF_CLASSES, np.bincount(rows["cls"].astype(np.int64), minlength=14)[1:].tolist()))
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            count()
            emit()
        torch.cuda.synchronize()
    res["per_call_us"] = {ev.key: round(ev.device_time_total / ev.count, 1) for ev in prof.key_averages()
                          if "k_var" in ev.key or "Memcpy" in ev.key or "k_scan" in ev.key or "Memset" in ev.key}
    res["card_after"] = k1_bench.card()
    plan.close()
    g.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
