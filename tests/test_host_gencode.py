"""NCBI genetic codes without a device: the tables of magot_b200.gencode against an independent statement of them, argument
validation, and the test reference (gencode_ref) against the oracle."""
import numpy as np
import pytest

import coracle
import gencode_ref as ref
import magot_oracle as mo
from magot_b200 import gencode


def test_supported_ids():
    assert gencode.SUPPORTED == tuple(sorted(ref.DIFFS))


@pytest.mark.parametrize("code", sorted(ref.DIFFS))
def test_tables_equal_the_published_differences(code):
    assert gencode.TABLES[code] == ref.ncbi_string(code)
    assert gencode.library(code) == ref.library(code)
    assert gencode.codon64(code) == ref.table64(code).encode()
    assert gencode.stops(code) == sorted(ref.STOPS[code].split())
    assert sorted(c for c, a in gencode.library(code).items() if a == "*") == sorted(ref.STOPS[code].split())
    assert gencode.check(str(code)) == code


def test_codon64_byte_order():
    t2 = gencode.codon64(2)
    idx = lambda c: 16 * "ACGT".index(c[0]) + 4 * "ACGT".index(c[1]) + "ACGT".index(c[2])
    assert t2[idx("AGA")] == ord("*") and t2[idx("AGG")] == ord("*") and t2[idx("TGA")] == ord("W") and t2[idx("ATA")] == ord("M")
    assert gencode.codon64(1)[idx("TGA")] == ord("*") and gencode.codon64(1)[idx("ATG")] == ord("M")
    assert gencode.library(1) == mo.CODON_TABLE
    assert len({bytes(ref.table64(c).encode()) for c in ref.STOP_SET_CODES}) == len(ref.STOP_SET_CODES)
    assert len({" ".join(sorted(ref.STOPS[c].split())) for c in ref.DIFFS}) == len(ref.STOP_SET_CODES)


def test_no_stop_in_the_ac_alphabet():
    """The stop-free stretches of the GPU tests use A and C only: no supported code has a stop, forward or reverse
    complement, in {A,C}^3."""
    for code in gencode.SUPPORTED:
        for s in gencode.stops(code):
            assert set(s) - set("AC") and set(ref.revcomp(s.encode()).decode()) - set("AC"), (code, s)


@pytest.mark.parametrize("bad", [0, 7, 8, 15, 17, 18, 19, 20, 27, 28, 31, 32, 34, -1, "abc", "", "5x", "1.0", 2.5, None, True])
def test_unsupported_ids_raise(bad):
    with pytest.raises(ValueError, match="supported NCBI tables"):
        gencode.check(bad)
    with pytest.raises(ValueError):
        gencode.codon64(bad)


def test_api_validates_before_device_work(tmp_path):
    """Bad codes are refused by the Python API and the command line before anything touches a device (this runs without
    one)."""
    from magot_b200 import genome, genome_tools as gt, orfs
    with pytest.raises(ValueError):
        genome.Sequence("ATGAAA").translate(genetic_code=7)
    with pytest.raises(ValueError):
        genome.Sequence("ATGAAA").translate(library=gencode.library(2), genetic_code=2)
    with pytest.raises(ValueError):
        genome.Sequence("ATGAAA").get_orfs(genetic_code="x")
    with pytest.raises(ValueError):
        orfs.sixframe(None, 0, 1, genetic_code=27)
    fa = tmp_path / "x.fa"
    fa.write_text(">a\nACGT\n")
    for argv in (["gff2fasta", str(fa), str(fa), "seq_type=protein", "genetic_code=five"],
                 ["cds2pep", str(fa), "genetic_code=31"],
                 ["dna2orfs", str(fa), str(tmp_path / "o.fa"), "genetic_code=8"]):
        with pytest.raises(ValueError):
            gt.main(["genome_tools.py"] + argv)
    assert not (tmp_path / "o.fa").exists()


def _random_seqs(rng, n):
    alpha = np.frombuffer(b"ACGTACGTACGTacgtNnRYKMSW-", dtype=np.uint8)
    return [alpha[rng.integers(0, alpha.size, size=int(k))].tobytes() for k in rng.integers(0, 200, size=n)]


@pytest.mark.parametrize("code", sorted(ref.DIFFS))
def test_reference_translate_equals_oracle(code):
    rng = np.random.default_rng(code)
    lib = gencode.library(code)
    for s in _random_seqs(rng, 60):
        for frame in (0, 1, 2):
            for minus in (False, True):
                for trim in (True, False):
                    want = mo.translate(s.decode(), frame=frame, strand='-' if minus else '+', trimX=trim, library=lib)
                    got = ref.translate(s, gencode.codon64(code).decode(), frame, minus, trim)
                    assert got == (None if want is None else want.encode()), (code, s, frame, minus, trim)


@pytest.mark.parametrize("code", sorted(ref.DIFFS))
def test_reference_orfs_equal_oracle(code):
    rng = np.random.default_rng(100 + code)
    lib = gencode.library(code)
    for s in _random_seqs(rng, 40):
        want = ref.get_orfs(s.decode(), lib)
        aa, recs = ref.sixframe(s, 0, gencode.codon64(code).decode())
        got = [aa[sum(r[3] for r in recs[:i]):][:r[3]].decode() for i, r in enumerate(recs)]
        assert got == want
        if code == 1:
            assert want == mo.get_orfs(s.decode())
            for min_aa in (0, 3):
                caa, crec = coracle.sixframe(s, min_aa)
                raa, rrec = ref.sixframe(s, min_aa, gencode.codon64(1).decode())
                assert caa == raa and [tuple(int(v) for v in r) for r in crec] == rrec
