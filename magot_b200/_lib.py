"""ctypes binding of libmagot_b200.so (C ABI declared in include/magot_b200.h).

There is no CPU fallback: if the shared library has not been built, importing this module
raises, and every compute entry point raises `MagotError` when no CUDA device is present.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# MAGOT_B200_LIB: developer knob for A/B runs of differently compiled builds of the same sources (scratch/variants.sh)
LIB_PATH = os.environ.get("MAGOT_B200_LIB") or os.path.join(_HERE, "libmagot_b200.so")

MG_PROT_TRIMX = 1
MG_PROT_USE_PHASE = 2
MG_PROT_DEFER = 4
MG_PRED_5PARTIAL = 1
MG_PRED_3PARTIAL = 2


class MagotError(RuntimeError):
    """An mg_* call returned a non-zero status."""


class MgOrf(ctypes.Structure):
    """mg_orf (include/magot_b200.h)."""
    _fields_ = [("contig", ctypes.c_int32), ("frame", ctypes.c_int8), ("minus", ctypes.c_int8),
                ("pad", ctypes.c_int16), ("start", ctypes.c_int64), ("len", ctypes.c_int64),
                ("aa_off", ctypes.c_int64)]


class MgOrfCall(ctypes.Structure):
    """mg_orfcall (include/magot_b200.h)."""
    _fields_ = [("contig", ctypes.c_int32), ("minus", ctypes.c_int8), ("phase", ctypes.c_int8),
                ("flags", ctypes.c_int8), ("start_codon", ctypes.c_int8), ("lo", ctypes.c_int64),
                ("hi", ctypes.c_int64), ("len", ctypes.c_int64), ("aa_off", ctypes.c_int64)]


class MgCdsCheck(ctypes.Structure):
    """mg_cds_check (include/magot_b200.h)."""
    _fields_ = [("nuc_len", ctypes.c_int64), ("gc", ctypes.c_int64), ("n_codons", ctypes.c_int32),
                ("n_ambig", ctypes.c_int32), ("n_stop", ctypes.c_int32), ("first_stop", ctypes.c_int32),
                ("gc3", ctypes.c_int32), ("n_junction", ctypes.c_int32), ("n_noncanonical", ctypes.c_int32),
                ("flags", ctypes.c_int32), ("skip", ctypes.c_int8), ("rem", ctypes.c_int8), ("start_codon", ctypes.c_uint8),
                ("stop_codon", ctypes.c_uint8), ("pad", ctypes.c_int32)]


class MgCdsPred(ctypes.Structure):
    """mg_cds_pred (include/magot_b200.h)."""
    _fields_ = [("lo", ctypes.c_int64), ("hi", ctypes.c_int64), ("n_aa", ctypes.c_int32), ("frame", ctypes.c_int8),
                ("type", ctypes.c_int8), ("start_codon", ctypes.c_uint8), ("stop_codon", ctypes.c_uint8),
                ("n_cds_seg", ctypes.c_int32), ("pad", ctypes.c_int32)]


class MgCdsSeg(ctypes.Structure):
    """mg_cds_seg (include/magot_b200.h)."""
    _fields_ = [("lo", ctypes.c_int64), ("hi", ctypes.c_int64), ("phase", ctypes.c_int8), ("pad", ctypes.c_int8 * 7)]


#: orf_type text of mg_cds_pred.type (bit 0: 5' partial, bit 1: 3' partial)
ORF_TYPES = ("complete", "5prime_partial", "3prime_partial", "internal")

#: MG_CHK_* flag bits of mg_cds_check.flags, in bit order (the names genome_tools check_cds prints)
CHK_FLAGS = ("NO_START", "NO_STOP", "INTERNAL_STOP", "PARTIAL_CODON", "NONCANONICAL_SPLICE", "AMBIGUOUS", "EMPTY")

if not os.path.isfile(LIB_PATH):
    raise ImportError(
        "magot_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback." % LIB_PATH)

lib = ctypes.CDLL(LIB_PATH)

_vp = ctypes.c_void_p
_i64 = ctypes.c_int64
_i32 = ctypes.c_int
_pp = ctypes.POINTER(ctypes.c_void_p)
_pi64 = ctypes.POINTER(ctypes.c_int64)

#: every symbol include/magot_b200.h declares: (restype, argtypes)
SIGNATURES = {
    "mg_version": (_i32, []),
    "mg_last_error": (ctypes.c_char_p, []),
    "mg_device_count": (_i32, [ctypes.POINTER(ctypes.c_int)]),
    "mg_genome_create": (_i32, [_i32, _i64, _vp, _pp]),
    "mg_genome_pack": (_i32, [_vp, _i64, _i64, _vp, _i64, _vp]),
    "mg_genome_pack_device": (_i32, [_vp, _i64, _i64, _vp, _i64, _vp]),
    "mg_genome_pack_fasta": (_i32, [_vp, _i64, _vp, _i64, _vp]),
    "mg_count_line_ends": (_i32, [ctypes.c_char_p, _i64, _i64, _vp, _vp, _vp]),
    "mg_genome_finalize": (_i32, [_vp, _pi64]),
    "mg_genome_destroy": (_i32, [_vp]),
    "mg_genome_bytes": (_i64, [_vp]),
    "mg_genome_at_flags": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp]),
    "mg_window_sums": (_i32, [_i32, _vp, _i32, _i64, _i64, _i64, _i64, _vp, _vp]),
    "mg_genome_fetch": (_i32, [_vp, _i64, _i64, _i64, _i32, _vp, _vp]),
    "mg_plan_create": (_i32, [_vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _pp]),
    "mg_plan_destroy": (_i32, [_vp]),
    "mg_genome_mask": (_i32, [_vp, _i64, _vp, _vp, _vp, _i32, _i32, _vp]),
    "mg_plan_prepare": (_i32, [_vp, _i32, _pi64, _pi64, _vp]),
    "mg_plan_prepare_async": (_i32, [_vp, _i32, _i64, _i64, _vp]),
    "mg_plan_prepare_prot_async": (_i32, [_vp, _vp]),
    "mg_plan_totals": (_i32, [_vp, _pi64, _pi64, _vp]),
    "mg_plan_lengths": (_i32, [_vp, _vp, _vp, _vp]),
    "mg_plan_set_codon_table": (_i32, [_vp, _vp]),
    "mg_emit_nuc_device": (_i32, [_vp, _vp, _vp]),
    "mg_emit_prot_device": (_i32, [_vp, _vp, _vp]),
    "mg_emit_nuc_prot_device": (_i32, [_vp, _vp, _vp, _vp]),
    "mg_emit_nuc_prot_host": (_i32, [_vp, _vp, _vp, _vp]),
    "mg_emit_products_device": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "mg_emit_products_host": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "mg_emit_nuc_host": (_i32, [_vp, _vp, _vp]),
    "mg_emit_prot_host": (_i32, [_vp, _vp, _vp]),
    "mg_revcomp": (_i32, [_i32, _vp, _i64, _vp, _vp]),
    "mg_translate_ascii": (_i32, [_i32, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _i64, _vp, _vp, _vp]),
    "mg_translate_ascii_table": (_i32, [_i32, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _i64, _vp, _vp, _vp]),
    "mg_sixframe_count": (_i32, [_vp, _i64, _i64, _i64, _pi64, _pi64, _vp]),
    "mg_sixframe_count_list": (_i32, [_vp, _i64, _vp, _i64, _pi64, _pi64, _vp]),
    "mg_sixframe_count_table": (_i32, [_vp, _i64, _i64, _i64, _vp, _pi64, _pi64, _vp]),
    "mg_sixframe_count_list_table": (_i32, [_vp, _i64, _vp, _i64, _vp, _pi64, _pi64, _vp]),
    "mg_sixframe_emit": (_i32, [_vp, _vp, _vp, _vp]),
    "mg_sixframe_emit_device": (_i32, [_vp, _vp, _vp, _vp]),
    "mg_orfcall_count": (_i32, [_vp, _i64, _vp, _i64, _vp, _vp, _i32, _pi64, _pi64, _vp]),
    "mg_orfcall_emit": (_i32, [_vp, _vp, _vp, _vp]),
    "mg_orfcall_emit_device": (_i32, [_vp, _vp, _vp, _vp]),
    "mg_plan_check": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "mg_plan_check_device": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "mg_plan_predict_cds": (_i32, [_vp, _i64, _vp, _i32, _vp, _vp, _vp]),
    "mg_plan_predict_cds_device": (_i32, [_vp, _i64, _vp, _i32, _vp, _vp, _vp]),
    "mg_stream_sync": (_i32, [_i32, _vp]),
    "mg_copy_d2h_async": (_i32, [_i32, _vp, _vp, _i64, _vp]),
    "mg_tune": (_i32, [ctypes.c_char_p, _i32]),
    "mg_gff_parse": (_i32, [ctypes.c_char_p, _i64, ctypes.c_char_p, _i64, _pp]),
    "mg_gff_destroy": (_i32, [_vp]),
    "mg_gff_info": (_i32, [_vp, _vp]),
    "mg_gff_column": (_i32, [_vp, ctypes.c_char_p, _pp, _pi64, ctypes.POINTER(ctypes.c_int32)]),
    "mg_gff_strings": (_i32, [_vp, _vp, _i64, _vp, _i64, _vp]),
    "mg_gff_find": (_i64, [_vp, ctypes.c_char_p, _i64]),
    "mg_py2_order": (_i32, [_vp, _vp, _i64, _i32, _vp]),
    "mg_gff_py2_order": (_i32, [_vp, _vp, _i64, _i32, _vp]),
    "mg_gff_flatten": (_i32, [_vp, _vp, _i64, _vp, _i64, _i32, _pp]),
    "mg_gff_flat_destroy": (_i32, [_vp]),
    "mg_gff_flat_column": (_i32, [_vp, ctypes.c_char_p, _pp, _pi64, ctypes.POINTER(ctypes.c_int32)]),
    "mg_graph_begin": (_i32, [_i32, _vp]),
    "mg_graph_end": (_i32, [_i32, _vp, _pp]),
    "mg_graph_launch": (_i32, [_i32, _vp, _vp]),
    "mg_graph_destroy": (_i32, [_vp]),
    "mg_stream_wait_stream": (_i32, [_i32, _vp, _vp]),
    "mg_kernel_launches": (_i64, []),
}

for _name, (_res, _args) in SIGNATURES.items():
    _f = getattr(lib, _name)          # AttributeError here == the library does not export the ABI
    _f.restype = _res
    _f.argtypes = _args


def last_error():
    return (lib.mg_last_error() or b"").decode("latin-1")


def check(rc):
    if rc != 0:
        raise MagotError("libmagot_b200 error %d: %s" % (rc, last_error()))


def device_count():
    n = ctypes.c_int(0)
    rc = lib.mg_device_count(ctypes.byref(n))
    return n.value if rc == 0 else 0


def require_device(device=0):
    n = device_count()
    if device >= n:
        raise MagotError("CUDA device %d not available (%d visible). magot_b200 runs the sequence path on "
                         "a B200 only; there is no CPU fallback." % (device, n))
