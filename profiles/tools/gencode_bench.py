"""Genetic codes on the bench genome: config-5 six-frame scan (count + emit, min ORF 100 aa) under codes 1, 2, 6 and 23 --
including the one-time stop-index build each non-standard stop set costs -- and the config-4 CDS protein emit (K3, K23) with
code 1 vs code 5.  One JSON line; CUDA events, medians after warm-up.

    python profiles/tools/gencode_bench.py [--runs 21]      (MAGOT_BENCH_GENOME_BP overrides the 3.1 Gbp genome)
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))   # repo root
import numpy as np
import torch

from magot_b200 import _lib, engine, gencode, synth

GENOME_BP = int(os.environ.get("MAGOT_BENCH_GENOME_BP", 3_100_000_000))
N_TX = 200_000
SEED = 4


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=21)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    lib = _lib.lib
    _lib.require_device(0)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)
    ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731

    layout = synth.contig_layout("human", GENOME_BP, SEED)
    g = engine.DeviceGenome([l for _, l in layout], device=0)
    CH = 256 << 20
    for ci, (_, L) in enumerate(layout):
        for off in range(0, L, CH):
            n = min(CH, L - off)
            a = synth.synth_contig_device(n, SEED * 1000003 + ci * 64 + off // CH, dev)
            torch.cuda.synchronize()
            g.pack_device(ci, a.data_ptr(), n, offset=off, stream=sp)
            torch.cuda.synchronize()
            del a
    g.finalize()
    torch.cuda.empty_cache()
    out = {"card": card(), "genome_bp": GENOME_BP, "runs": args.runs}

    # ---- config 5 under four codes
    ids = np.arange(len(layout), dtype=np.int64)
    n_orf, n_bytes = ctypes.c_int64(0), ctypes.c_int64(0)
    six = {}
    for code in (1, 2, 6, 23):
        t = None if code == 1 else gencode.codon64(code)

        def count():
            _lib.check(lib.mg_sixframe_count_list_table(g.handle, ids.size, ctypes.c_void_p(ids.ctypes.data), 100, t,
                                                        ctypes.byref(n_orf), ctypes.byref(n_bytes), sp))
        b0 = g.device_bytes()
        torch.cuda.synchronize()
        f0, f1 = ev(), ev()
        f0.record(stream)
        count()                                          # builds this stop set's index (code 2 / 6 / 23: replaces the previous one)
        f1.record(stream)
        torch.cuda.synchronize()
        first = f0.elapsed_time(f1)
        aa = torch.empty((n_bytes.value + 31) // 32 * 32 + 32, dtype=torch.uint8, device=dev)
        scans, emits, tot = [], [], []
        for k in range(args.warmup + args.runs):
            a0, a1, a2 = ev(), ev(), ev()
            a0.record(stream)
            count()
            a1.record(stream)
            _lib.check(lib.mg_sixframe_emit_device(g.handle, ctypes.c_void_p(aa.data_ptr()), None, sp))
            a2.record(stream)
            torch.cuda.synchronize()
            if k >= args.warmup:
                scans.append(a0.elapsed_time(a1))
                emits.append(a1.elapsed_time(a2))
                tot.append(a0.elapsed_time(a2))
        six[str(code)] = {"orfs": n_orf.value, "aa_bytes": n_bytes.value, "count_ms": round(float(np.median(scans)), 3),
                          "emit_ms": round(float(np.median(emits)), 3), "count_plus_emit_ms": round(float(np.median(tot)), 3),
                          "count_plus_emit_min_max_ms": [round(min(tot), 3), round(max(tot), 3)],
                          "first_count_ms_incl_index_build": round(first, 3),
                          "stops": gencode.stops(code), "device_bytes_added": g.device_bytes() - b0}
        del aa
    out["config5_sixframe_min_aa_100"] = six

    # ---- config 4: CDS protein text (framed records), K3 and K23, code 1 vs code 5
    ann = synth.synth_annotation(layout, N_TX, SEED)
    tbl = ann.table("cds")
    emit = {}
    for code in (1, 5, 1, 5):                            # alternated, so drift of the shared host shows in both
        plan = engine.Plan(g, tbl, stream=sp)
        if code != 1:
            plan.set_codon_table(gencode.codon64(code))
        nt, pt = plan.prepare()
        on = torch.empty((nt + 31) // 32 * 32 + 32, dtype=torch.uint8, device=dev)
        op = torch.empty((pt + 31) // 32 * 32 + 32, dtype=torch.uint8, device=dev)
        res = {}
        for name, fn in (("k3_ms", lambda: lib.mg_emit_prot_device(plan.handle, ctypes.c_void_p(op.data_ptr()), sp)),
                         ("k23_ms", lambda: lib.mg_emit_nuc_prot_device(plan.handle, ctypes.c_void_p(on.data_ptr()),
                                                                         ctypes.c_void_p(op.data_ptr()), sp))):
            ts = []
            for k in range(args.warmup + args.runs):
                a0, a1 = ev(), ev()
                a0.record(stream)
                _lib.check(fn())
                a1.record(stream)
                torch.cuda.synchronize()
                if k >= args.warmup:
                    ts.append(a0.elapsed_time(a1))
            res[name] = round(float(np.median(ts)), 4)
        res["prot_bytes"] = pt
        res["prot_sum"] = int(op[:pt].to(torch.int64).sum().item())
        plan.close()
        emit.setdefault(str(code), []).append(res)
    out["config4_cds_protein_emit"] = emit
    g.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
