"""Start-to-stop ORF calling on the bench genome (config 5's 3.1 Gbp, min ORF 100 aa): mg_orfcall_count + mg_orfcall_emit_device
under codes 1 and 11 with {ATG} and {ATG, GTG, TTG}, and code 1 with 3' partials, interleaved in one process with the K4
six-frame count + emit under code 1 as the baseline.  One JSON line; CUDA events, medians after warm-up.

    python profiles/tools/orfcall_bench.py [--runs 21] [--warmup 3]      (MAGOT_BENCH_GENOME_BP overrides the 3.1 Gbp genome)
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
SEED = 4
MIN_AA = 100
CASES = (("code1_atg", 1, ("ATG",), 0), ("code1_atg_gtg_ttg", 1, ("ATG", "GTG", "TTG"), 0), ("code11_atg", 11, ("ATG",), 0),
         ("code11_atg_gtg_ttg", 11, ("ATG", "GTG", "TTG"), 0), ("code1_atg_partial", 1, ("ATG",), 1))


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
    out = {"card": card(), "genome_bp": GENOME_BP, "min_aa": MIN_AA, "runs": args.runs, "warmup": args.warmup}

    ids = np.arange(len(layout), dtype=np.int64)
    idp = ctypes.c_void_p(ids.ctypes.data)
    n_orf, n_bytes = ctypes.c_int64(0), ctypes.c_int64(0)
    aa = {}

    def k4():
        _lib.check(lib.mg_sixframe_count_list_table(g.handle, ids.size, idp, MIN_AA, None, ctypes.byref(n_orf),
                                                    ctypes.byref(n_bytes), sp))
        return lambda buf: _lib.check(lib.mg_sixframe_emit_device(g.handle, ctypes.c_void_p(buf.data_ptr()), None, sp))

    def orfcall(code, starts, partial):
        t = None if code == 1 else gencode.codon64(code)
        s64 = gencode.start64(starts, code)

        def run():
            _lib.check(lib.mg_orfcall_count(g.handle, ids.size, idp, MIN_AA, t, s64, partial, ctypes.byref(n_orf),
                                            ctypes.byref(n_bytes), sp))
            return lambda buf: _lib.check(lib.mg_orfcall_emit_device(g.handle, ctypes.c_void_p(buf.data_ptr()), None, sp))
        return run

    runs = [("k4_sixframe_code1", k4)] + [(name, orfcall(code, starts, partial)) for name, code, starts, partial in CASES]
    res = {name: {"count_ms": [], "emit_ms": [], "total_ms": []} for name, _ in runs}
    for name, fn in runs:                                 # first call of each, in this order: the first one builds the stop index
        torch.cuda.synchronize()
        f0, f1 = ev(), ev()
        f0.record(stream)
        emit = fn()
        aa[name] = torch.empty((n_bytes.value + 31) // 32 * 32 + 32, dtype=torch.uint8, device=dev)
        emit(aa[name])
        f1.record(stream)
        torch.cuda.synchronize()
        res[name]["first_count_plus_emit_ms"] = round(f0.elapsed_time(f1), 3)
    for k in range(args.warmup + args.runs):             # interleaved: drift of the shared host shows in every case
        for name, fn in runs:
            a0, a1, a2 = ev(), ev(), ev()
            a0.record(stream)
            emit = fn()
            a1.record(stream)
            emit(aa[name])
            a2.record(stream)
            torch.cuda.synchronize()
            if k >= args.warmup:
                res[name]["count_ms"].append(a0.elapsed_time(a1))
                res[name]["emit_ms"].append(a1.elapsed_time(a2))
                res[name]["total_ms"].append(a0.elapsed_time(a2))
            res[name]["orfs"] = n_orf.value
            res[name]["aa_bytes"] = n_bytes.value
    base = float(np.median(res["k4_sixframe_code1"]["total_ms"]))
    for name, r in res.items():
        tot = r.pop("total_ms")
        r["count_ms"] = round(float(np.median(r["count_ms"])), 3)
        r["emit_ms"] = round(float(np.median(r["emit_ms"])), 3)
        r["count_plus_emit_ms"] = round(float(np.median(tot)), 3)
        r["count_plus_emit_min_max_ms"] = [round(min(tot), 3), round(max(tot), 3)]
        r["vs_k4"] = round(float(np.median(tot)) / base, 3)
    out["cases"] = res
    g.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
