"""The gene-model check against K3 on config 4's CDS plan: mg_plan_check_device in three forms (summary only, with the 64
codon counts per record, with the junction classes) and K3 alone (mg_emit_prot_device) on the same prepared plan, each timed
with CUDA events over REPS launches after WARM warm-up launches.  The genome and the table come from the seeds and generators
k1_bench.py uses.  Prints one JSON line with the card's name, power limit and SM clock read in the same run.

    python profiles/tools/check_bench.py [tag]          env: CKB_REPS (default 200), CKB_WARM (20), MAGOT_BENCH_TX (200000)
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
REPS = int(os.environ.get("CKB_REPS", 200))
WARM = int(os.environ.get("CKB_WARM", 20))
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
    t = synth.synth_annotation(layout, k1_bench.N_TX, k1_bench.SEED).table("cds")
    plan = engine.Plan(g, t, stream=sp)
    nuc_total, prot_total = plan.prepare()
    n, e = t.n_rec, t.n_seg
    d_rec = torch.empty(n * ctypes.sizeof(_lib.MgCdsCheck), dtype=torch.uint8, device=dev)
    d_cnt = torch.empty(n * 256, dtype=torch.uint8, device=dev)
    d_jn = torch.empty(max(e, 1), dtype=torch.uint8, device=dev)
    d_prot = torch.empty((prot_total + 31) // 32 * 32 + 32, dtype=torch.uint8, device=dev)
    P = lambda x: ctypes.c_void_p(x.data_ptr()) if x is not None else None   # noqa: E731

    def chk(counts, junction):
        return lambda: _lib.check(lib.mg_plan_check_device(plan.handle, 0, None, P(d_rec), P(counts), P(junction), sp))

    res = {"tag": tag, "card": k1_bench.card(), "reps": REPS, "n_tx": k1_bench.N_TX, "n_rec": int(n), "n_seg": int(e),
           "cds_bases": int(nuc_total), "residues": int(prot_total)}
    res["k3"] = k1_bench.timed(lambda: _lib.check(lib.mg_emit_prot_device(plan.handle, P(d_prot), sp)), stream)
    res["check_summary"] = k1_bench.timed(chk(None, None), stream)
    res["check_counts"] = k1_bench.timed(chk(d_cnt, None), stream)
    res["check_junctions"] = k1_bench.timed(chk(None, d_jn), stream)
    res["summary_over_k3"] = round(res["check_summary"]["ms_med"] / res["k3"]["ms_med"], 3)
    # per-kernel split of the summary-only check, from torch.profiler in a window of its own
    from torch.profiler import profile, ProfilerActivity
    f = chk(None, None)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            f()
        torch.cuda.synchronize()
    res["check_kernels_us"] = {ev.key: round(ev.device_time_total / ev.count, 1) for ev in prof.key_averages()
                               if ev.key.startswith(("k_check", "void k_check"))}
    rec = d_rec.cpu().numpy().view(engine.CHECK_DTYPE)
    res["flag_counts"] = [int(((rec["flags"] >> k) & 1).sum()) for k in range(7)]
    res["card_after"] = k1_bench.card()
    plan.close()
    g.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
