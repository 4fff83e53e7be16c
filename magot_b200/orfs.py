"""Host wrapper of K4 (six-frame translation + ORF scan on device-resident contigs).

Replaces Sequence.get_orfs (genome.py:824-851) applied to whole contigs -- what dna2orfs
(genome_tools.py:145-180) intended -- with an optional minimum length (0 == reference).
call_orfs() is start-to-stop ORF calling on the same scan (mg_orfcall_count): true phases, genome coordinates.
"""
import ctypes

import numpy as np

from . import _lib
from . import gencode
from ._lib import lib, check

ORF_DTYPE = np.dtype([("contig", np.int32), ("frame", np.int8), ("minus", np.int8), ("pad", np.int16),
                      ("start", np.int64), ("len", np.int64), ("aa_off", np.int64)])
assert ORF_DTYPE.itemsize == ctypes.sizeof(_lib.MgOrf)

ORFCALL_DTYPE = np.dtype([("contig", np.int32), ("minus", np.int8), ("phase", np.int8), ("flags", np.int8),
                          ("start_codon", np.int8), ("lo", np.int64), ("hi", np.int64), ("len", np.int64),
                          ("aa_off", np.int64)])
assert ORFCALL_DTYPE.itemsize == ctypes.sizeof(_lib.MgOrfCall)


def _codon64(genetic_code):
    code = gencode.check(genetic_code)
    return None if code == 1 else gencode.codon64(code)


def sixframe(device_genome, contig_lo, contig_hi, min_aa=0, stream=None, genetic_code=1):
    """ORFs of contigs [contig_lo, contig_hi) in reference order, translated with NCBI table `genetic_code` and split
    on its stops.  Returns (records: structured array ORF_DTYPE, residues: bytes with the ORFs back to back)."""
    table = _codon64(genetic_code)
    n_orf, n_bytes = ctypes.c_int64(0), ctypes.c_int64(0)
    check(lib.mg_sixframe_count_table(device_genome.handle, contig_lo, contig_hi, int(min_aa), table,
                                      ctypes.byref(n_orf), ctypes.byref(n_bytes), stream))
    recs = np.zeros(n_orf.value, dtype=ORF_DTYPE)
    aa = np.empty(max(n_bytes.value, 1), dtype=np.uint8)
    check(lib.mg_sixframe_emit(device_genome.handle, ctypes.c_void_p(aa.ctypes.data),
                               ctypes.c_void_p(recs.ctypes.data) if n_orf.value else None, stream))
    check(lib.mg_stream_sync(device_genome.device, stream))
    return recs, aa[:n_bytes.value].tobytes()


def sixframe_list(device_genome, contig_ids, min_aa=0, stream=None, genetic_code=1):
    """ORFs of the listed contigs (any order), contig by contig in list order; same arguments and return as sixframe()."""
    table = _codon64(genetic_code)
    ids = np.ascontiguousarray(contig_ids, dtype=np.int64)
    n_orf, n_bytes = ctypes.c_int64(0), ctypes.c_int64(0)
    check(lib.mg_sixframe_count_list_table(device_genome.handle, ids.size, ctypes.c_void_p(ids.ctypes.data), int(min_aa),
                                           table, ctypes.byref(n_orf), ctypes.byref(n_bytes), stream))
    recs = np.zeros(n_orf.value, dtype=ORF_DTYPE)
    aa = np.empty(max(n_bytes.value, 1), dtype=np.uint8)
    check(lib.mg_sixframe_emit(device_genome.handle, ctypes.c_void_p(aa.ctypes.data),
                               ctypes.c_void_p(recs.ctypes.data) if n_orf.value else None, stream))
    check(lib.mg_stream_sync(device_genome.device, stream))
    return recs, aa[:n_bytes.value].tobytes()


def call_orfs(device_genome, contig_ids, min_aa=100, genetic_code=1, start_codons=("ATG",), partial=False, stream=None):
    """Start-to-stop ORFs of the listed contigs on both strands and all three phases (include/magot_b200.h, mg_orfcall):
    each stop-bounded stretch gives the ORF from its first start codon through the stop, of >= min_aa residues ('M'
    included, stop excluded); partial=True adds those that reach the contig end without a stop (flags bit 0).
    Returns (records: structured array ORFCALL_DTYPE in the ABI's order, residues: bytes with the proteins back to back)."""
    table = _codon64(genetic_code)
    starts = gencode.start64(start_codons, genetic_code)
    ids = np.ascontiguousarray(contig_ids, dtype=np.int64)
    n_orf, n_bytes = ctypes.c_int64(0), ctypes.c_int64(0)
    check(lib.mg_orfcall_count(device_genome.handle, ids.size, ctypes.c_void_p(ids.ctypes.data), int(min_aa), table, starts,
                               1 if partial else 0, ctypes.byref(n_orf), ctypes.byref(n_bytes), stream))
    recs = np.zeros(n_orf.value, dtype=ORFCALL_DTYPE)
    aa = np.empty(max(n_bytes.value, 1), dtype=np.uint8)
    check(lib.mg_orfcall_emit(device_genome.handle, ctypes.c_void_p(aa.ctypes.data),
                              ctypes.c_void_p(recs.ctypes.data) if n_orf.value else None, stream))
    check(lib.mg_stream_sync(device_genome.device, stream))
    return recs, aa[:n_bytes.value].tobytes()


def lpt_shards(lengths, n_shards):
    """Longest-processing-time assignment of contigs to n_shards GPUs: shards[i] = contig indices (ascending) of GPU i."""
    order = np.argsort(-np.asarray(lengths, dtype=np.int64), kind="stable")
    load = [0] * n_shards
    shards = [[] for _ in range(n_shards)]
    for c in order:
        k = min(range(n_shards), key=lambda i: load[i])
        shards[k].append(int(c))
        load[k] += int(lengths[c])
    return [sorted(x) for x in shards]


def contig_orfs(genome_sequence, seqid, min_aa=0, genetic_code=1):
    """(records, list of ORF strings) for one contig of a magot_b200.genome.GenomeSequence."""
    ci = genome_sequence.contig_index(seqid)
    recs, aa = sixframe(genome_sequence._engine().primary, ci, ci + 1, min_aa, genetic_code=genetic_code)
    text = aa.decode("latin-1")
    out = [text[int(r["aa_off"]):int(r["aa_off"]) + int(r["len"])] for r in recs]
    return recs, out
