"""K1 alone: each plan pass of config 4 timed with CUDA events, at the full batch and at its first eighth of the records
(about the shard one rank of 8 gets in bench.py's strong scaling).

For the CDS and the exon table: the piece pass (mg_plan_prepare_async with MG_PROT_DEFER, i.e. the look-back memset and
k_plan_pieces) and, for CDS, the record pass (mg_plan_prepare_prot_async: memset and k_plan_records), each alone on one
stream; also both passes in series as bench.py's kernel table times them.  Median and min of REPS launches after WARM
warm-up launches.  Prints one JSON line with the card's name, power limit and SM clock read in the same run.

    python profiles/tools/k1_bench.py [tag]          env: K1B_REPS (default 200), K1B_WARM (20), MAGOT_BENCH_TX (200000)
"""
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))   # repo root
import numpy as np
import torch

from magot_b200 import _lib, engine, synth

lib = _lib.lib
GENOME_BP = int(os.environ.get("MAGOT_BENCH_GENOME_BP", 3_100_000_000))
SEED = 4
N_TX = int(os.environ.get("MAGOT_BENCH_TX", 200_000))
REPS = int(os.environ.get("K1B_REPS", 200))
WARM = int(os.environ.get("K1B_WARM", 20))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return [s.strip() for s in q.split(",")]
    except Exception as e:                             # the numbers are still measured; say why the card is not named
        return ["unknown: %s" % e]


def timed(fn, stream):
    for _ in range(WARM):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(REPS)]
    for a, b in ev:
        a.record(stream)
        fn()
        b.record(stream)
    torch.cuda.synchronize()
    t = np.array([a.elapsed_time(b) for a, b in ev])
    return {"ms_med": round(float(np.median(t)), 4), "ms_min": round(float(t.min()), 4)}


def main():
    tag = sys.argv[1] if len(sys.argv) > 1 else ""
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)
    layout = synth.contig_layout("human", GENOME_BP, SEED)
    g = engine.DeviceGenome([n for _, n in layout], device=0)
    CH = 256 << 20
    for ci, (_, L) in enumerate(layout):
        for off in range(0, L, CH):
            n = min(CH, L - off)
            a = synth.synth_contig_device(n, SEED * 1000003 + ci * 64 + off // CH, dev)
            g.pack_device(ci, a.data_ptr(), n, offset=off, stream=sp)
            torch.cuda.synchronize()
            del a
    g.finalize()
    torch.cuda.empty_cache()
    ann_all = synth.synth_annotation(layout, N_TX, SEED)
    res = {"tag": tag, "card": card(), "reps": REPS, "n_tx": N_TX}
    flags = _lib.MG_PROT_TRIMX
    for name, ann in (("full", ann_all), ("eighth", ann_all.subset(np.arange(0, N_TX // 8)))):
        out = {}
        for which in ("cds", "exon"):
            t = ann.table(which)
            plan = engine.Plan(g, t, stream=sp)
            cap_n, cap_p = plan.capacities()
            h = plan.handle
            piece = lambda: _lib.check(lib.mg_plan_prepare_async(h, flags | _lib.MG_PROT_DEFER, cap_n, cap_p, sp))   # noqa: E731
            piece()
            torch.cuda.synchronize()
            r = {"n_rec": int(t.n_rec), "n_piece": int(t.n_seg + 2 * t.n_rec), "piece_pass": timed(piece, stream)}
            if which == "cds":
                def rec_timed():                       # a record pass runs once per piece pass: re-arm it outside the window
                    ev = []
                    for i in range(WARM + REPS):
                        piece()
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record(stream)
                        _lib.check(lib.mg_plan_prepare_prot_async(h, sp))
                        b.record(stream)
                        ev.append((a, b))
                    torch.cuda.synchronize()
                    x = np.array([a.elapsed_time(b) for a, b in ev[WARM:]])
                    return {"ms_med": round(float(np.median(x)), 4), "ms_min": round(float(x.min()), 4)}
                r["record_pass"] = rec_timed()
                both = lambda: _lib.check(lib.mg_plan_prepare_async(h, flags, cap_n, cap_p, sp))   # noqa: E731
                r["both_passes"] = timed(both, stream)
            plan.close()
            out[which] = r
        res[name] = out
    res["card_after"] = card()
    g.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
