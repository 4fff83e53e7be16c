"""CDS prediction against K2 on config 4's exon plan: mg_plan_predict_cds_device sense-only in three forms (records only,
records with both partial flags, records and the per-segment CDS coordinates) and K2 alone (mg_emit_nuc_device) on the same plan
after a deferred prepare (the piece pass only, as AnnotationSet.predict_cds runs it), each timed with CUDA events over REPS
launches after WARM warm-up launches, and a torch.profiler split per kernel.  The genome and the table come from the seeds and
generators k1_bench.py uses.  Prints one JSON line with the card's name, power limit and SM clock read in the same run.

    python profiles/tools/predict_bench.py [tag]        env: PRB_REPS (default 200), PRB_WARM (20), MAGOT_BENCH_TX (200000)
"""
import ctypes
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))   # repo root
import numpy as np
import torch

from magot_b200 import _lib, engine, synth
import k1_bench

lib = _lib.lib
REPS = int(os.environ.get("PRB_REPS", 200))
WARM = int(os.environ.get("PRB_WARM", 20))
k1_bench.REPS, k1_bench.WARM = REPS, WARM


def main():
    tag = sys.argv[1] if len(sys.argv) > 1 else ""
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)
    layout = synth.contig_layout("human", k1_bench.GENOME_BP, k1_bench.SEED)
    g = engine.DeviceGenome([n for _, n in layout], device=0)
    CH = 256 << 20
    for ci, (_, L) in enumerate(layout):
        for off in range(0, L, CH):
            n = min(CH, L - off)
            a = synth.synth_contig_device(n, k1_bench.SEED * 1000003 + ci * 64 + off // CH, dev)
            g.pack_device(ci, a.data_ptr(), n, offset=off, stream=sp)
            torch.cuda.synchronize()
            del a
    g.finalize()
    torch.cuda.empty_cache()
    t = synth.synth_annotation(layout, k1_bench.N_TX, k1_bench.SEED).table("exon")
    plan = engine.Plan(g, t, stream=sp)
    cap_n, _ = plan.prepare_async(defer_records=True)
    torch.cuda.synchronize()
    n, e = t.n_rec, t.n_seg
    d_rec = torch.empty(n * ctypes.sizeof(_lib.MgCdsPred), dtype=torch.uint8, device=dev)
    d_seg = torch.empty(max(e, 1) * ctypes.sizeof(_lib.MgCdsSeg), dtype=torch.uint8, device=dev)
    d_nuc = torch.empty((cap_n + 31) // 32 * 32 + 32, dtype=torch.uint8, device=dev)
    P = lambda x: ctypes.c_void_p(x.data_ptr()) if x is not None else None   # noqa: E731
    both = _lib.MG_PRED_5PARTIAL | _lib.MG_PRED_3PARTIAL

    def pred(flags, seg):
        return lambda: _lib.check(lib.mg_plan_predict_cds_device(plan.handle, 100, None, flags, P(d_rec), P(seg), sp))

    res = {"tag": tag, "card": k1_bench.card(), "reps": REPS, "n_tx": k1_bench.N_TX, "n_rec": int(n), "n_seg": int(e)}
    res["k2"] = k1_bench.timed(lambda: _lib.check(lib.mg_emit_nuc_device(plan.handle, P(d_nuc), sp)), stream)
    res["predict"] = k1_bench.timed(pred(0, None), stream)
    res["predict_partial"] = k1_bench.timed(pred(both, None), stream)
    res["predict_segments"] = k1_bench.timed(pred(0, d_seg), stream)
    res["predict_over_k2"] = round(res["predict"]["ms_med"] / res["k2"]["ms_med"], 3)
    res["predict_segments_over_k2"] = round(res["predict_segments"]["ms_med"] / res["k2"]["ms_med"], 3)
    from torch.profiler import profile, ProfilerActivity
    f = pred(0, d_seg)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            f()
        torch.cuda.synchronize()
    res["predict_kernels_us"] = {ev.key: round(ev.device_time_total / ev.count, 1) for ev in prof.key_averages()
                                 if "k_predict" in ev.key}
    nuc_total, _ = plan.totals()
    rec = d_rec.cpu().numpy().view(engine.PRED_DTYPE)
    res["exon_bases"] = int(nuc_total)
    res["with_orf"] = int((rec["n_aa"] > 0).sum())
    res["median_aa"] = float(np.median(rec["n_aa"][rec["n_aa"] > 0])) if res["with_orf"] else 0.0
    res["card_after"] = k1_bench.card()
    plan.close()
    g.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
