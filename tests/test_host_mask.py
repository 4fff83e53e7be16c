"""The byte model genome_model (what tests/test_gpu_mask.py compares the device with), checked without a GPU: its
mask_from_gff against the reference's own output (manifest.json cksums, written by tests/golden/make_golden.py) and its
genome operations on hand-written cases."""
import os

import numpy as np
import pytest

import genome_model as gm
from cksum import cksum

INPUTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "aligner_inputs")


def _read(path, binary=False):
    with open(path, "rb") as fh:
        data = fh.read()
    return data if binary else data.decode("latin-1")


def _ck(text):
    c, n = cksum(text)
    return {"cksum": c, "bytes": n}


def test_model_mask_from_gff_matches_reference(ref_data, manifest):
    fa = _read(os.path.join(INPUTS, "mask.fasta"), binary=True)
    gff, gff_soft = _read(os.path.join(INPUTS, "mask.gff")), _read(os.path.join(INPUTS, "mask_soft.gff"))
    ob_fa = _read(os.path.join(ref_data, "O.biroi_refseqGenomeSubset.fasta"), binary=True)
    ob_gff = _read(os.path.join(ref_data, "O.biroi_NCBIrefseq_gff3Subset.gff"))
    assert _ck(gm.mask_from_gff(fa, gff_soft)) == manifest["mask:soft"]
    assert _ck(gm.mask_from_gff(fa, gff_soft, overwrite_softmask="False")) == manifest["mask:soft_keep_case"]
    assert _ck(gm.mask_from_gff(fa, gff, mask_type="hard")) == manifest["mask:hard"]
    assert _ck(gm.mask_from_gff(fa, gff, "hard", "F", "exon")) == manifest["mask:hard_keep_case_exon"]
    assert _ck(gm.mask_from_gff(ob_fa, ob_gff)) == manifest["mask:obiroi_soft"]
    assert _ck(gm.mask_from_gff(ob_fa, ob_gff, "hard", "False", "exon")) == manifest["mask:obiroi_hard_exon"]
    with pytest.raises(NotImplementedError):               # the reference would lengthen the sequence here
        gm.mask_from_gff(fa, gff_soft, mask_type="hard")


def test_model_mask_from_gff_hand_cases():
    fa = b">b desc\r\nACGTRYKMNn\r\nacgtW*\n>a\nAAAA\n>b\nACGTACGTAC\n"     # b repeated: starts over
    line = "\t".join
    gff = "\n".join([line(["b", "s", "CDS", "0", "3", ".", "+", ".", "x\r"]),      # [-1:3] of 10 bases: empty
                     line(["b", "s", "CDS", "9", "3", ".", "+", ".", "x"]),        # reversed: empty
                     line(["b", "s", "CDS", "-2", "10", ".", "+", ".", "x"]),      # [-3:10]: the last 3 bases
                     line(["b", "s", "CDS", "2", "3", ".", "+"]),                  # 6 tabs: counts
                     line(["b", "s", "CDS", "4", "5", "."]),                       # 5 tabs: ignored
                     line(["a", "s", "exon", "1", "4", ".", "+", ".", "x"])]) + "\n"
    out = gm.mask_from_gff(fa, gff)
    recs = dict(zip(out.split(b"\n")[0:-1:2], out.split(b"\n")[1::2]))
    assert recs == {b">a": b"AAAA", b">b": b"AcgTACGtac"}
    out = gm.mask_from_gff(fa, gff.replace("CDS", "gene"), "hard", "False", "exon")
    assert b">a\nNNNN\n" in out and b">b\nACGTACGTAC\n" in out
    with pytest.raises(NotImplementedError):               # start = 0: [-1:3] is empty, 4 'N's would be written
        gm.mask_from_gff(fa, gff, "hard")


def test_model_genome_hand_cases():
    g = gm.Genome([b"ACGTRYKMNn-acgtrW*\xe9 ", b"", b"aTtA"])
    assert g.n_exceptions() == 5                            # r W * \xe9 and the space
    assert g.fetch(0, 0, 4, minus=True) == b"ACGT"
    assert g.fetch(0, 4, 11, minus=True) == b"-nNnnnn"
    g.mask([0, 0], [0, 2], [6, 8])                          # soft, overlapping: R Y K M -> r y k m, listed
    assert g.fetch(0, 0, 10) == b"acgtrykmNn" and g.n_exceptions() == 9
    g.mask([0], [16], [19], upper_first=True)               # upper first: listed bytes stay listed
    assert g.fetch(0, 0, 19) == b"ACGTRYKMNN-ACGTRw*\xe9" and g.n_exceptions() == 9
    g.mask([0, 2], [3, 1], [5, 3], hard=True)
    assert g.fetch(0, 0, 8) == b"ACGNNYKM" and g.n_exceptions() == 8
    assert g.fetch(2, 0, 4) == b"ANNA"
    assert np.array_equal(g.at_flags(2, 0, 4), [1, 0, 0, 1])
    assert np.array_equal(gm.at_flags(b"ATatNnRrWw"), [1, 1, 1, 1, 0, 0, 0, 0, 0, 0])
