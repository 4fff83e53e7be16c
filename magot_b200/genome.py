"""Drop-in mirror of the sequence half of MAGOT's `genome` module (reference: genome.py).

Same names, signatures, return types and text output as the reference for the
annotation-driven sequence path; underneath, the genome is packed once into a device-resident
nibble buffer, annotations are flattened on the host into SoA interval tables and the
extraction / reverse-complement / translation run as sm_100a CUDA kernels behind the C ABI in
include/magot_b200.h.  There is no CPU fallback for any of that work.

Reference API kept (file:line in /root/reference/genome.py):
  Sequence(str)            :781   reverse_compliment :784, translate :795, get_orfs :824
  GenomeSequence           :854   dict-like seqid -> contig (values are lazy device views)
  Genome                   :880   ctor :883, get_scaffold_fasta :907, get_genome_fasta :910,
                                   get_seqids :935, read_gff :970
  read_gff                 :242   (presets= is not supported: it relies on py2 `exec` semantics)
  AnnotationSet            :524   __getitem__ :536, read_gff :546, get_fasta :578
  BaseAnnotation           :586   get_coords :600, get_seq :603
  ParentAnnotation         :649   get_coords :663, get_fasta :677
Record order: the reference iterates Python-2.7 dicts; `RECORD_ORDER = "py2"` (default) replays
that order (magot_b200.py2dict) so whole files are byte-identical; "insertion" keeps file order.
"""
import collections
import io
import os

import numpy as np

from . import _lib
from . import engine
from . import gencode
from .py2dict import py2_order, py2_order_after_deepcopy, py2_instance_attr_order
import weakref

verbose = True                      # genome.py:22
RECORD_ORDER = "py2"                # "py2" (reference-identical) | "insertion"
DEFAULT_DEVICES = None              # None -> [0]; or a list of CUDA device indices to shard over
TIMINGS = None                      # a dict here receives the split of the last native get_fasta call (bench.py: api_e2e)


def _order(keys, deepcopy=False):
    if RECORD_ORDER != "py2":
        return list(keys)
    return py2_order_after_deepcopy(keys) if deepcopy else py2_order(keys)


# AnnotationSets that read_gff created itself: the reference returns copy.deepcopy of them (genome.py:415), which
# also changes the iteration order of every instance __dict__ (used by write_gff / "extended gff3").
_DEEPCOPIED_SETS = weakref.WeakSet()


def _attr_order(obj):
    """Attribute names of obj in the order a CPython-2.7 instance __dict__ would iterate them."""
    names = list(obj.__dict__)
    if RECORD_ORDER != "py2":
        return names
    aset = obj if isinstance(obj, AnnotationSet) else getattr(obj, "annotation_set", None)
    return py2_instance_attr_order(names, deepcopied=aset is not None and aset in _DEEPCOPIED_SETS)


def _py2_str(value):
    """str() as Python 2.7 prints it: floats with 12 significant digits (`score` column of get_gff)."""
    if isinstance(value, float):
        t = "%.12g" % value
        if "." not in t and "e" not in t and "n" not in t:      # 'inf' / 'nan' carry an 'n'
            t += ".0"
        return t
    return str(value)


def _gff_columns(obj):
    """The eight leading GFF columns of get_gff (genome.py:618-625 / :738-745): a missing attribute prints '.',
    anything else (e.g. get_coords() of a childless parent being None) raises like the reference's eval."""
    fields_list = []
    for field in ('seqid', 'source', 'feature_type', 0, 1, 'score', 'strand', 'phase'):
        try:
            if isinstance(field, int):
                fields_list.append(_py2_str(obj.get_coords()[field]))
            else:
                fields_list.append(_py2_str(getattr(obj, field)))
        except AttributeError:
            fields_list.append('.')
    return fields_list


_GFF3_FORMATS = ("simple gff3", "extended gff3", "exon added gff3")


def _gff_format_kind(gff_format):
    """'gff3' | 'hint' | 'gtf' | None (a format get_gff does not know: the reference then fails on an unbound local)."""
    if gff_format in _GFF3_FORMATS:
        return "gff3"
    if gff_format[:13] == "augustus hint":
        return "hint"
    return "gtf" if gff_format == "gtf" else None
_NOT_EXTENDED = ('ID', 'Parent', 'score', 'strand', 'seqid', 'feature_type', 'phase', 'source')


def _gff3_defline(obj, gff_format):
    """ID=..;Parent=.. (+ every other str attribute in instance-dict order for "extended gff3"), genome.py:626-633."""
    defline = 'ID=' + obj.ID
    if obj.parent is not None:
        defline = defline + ';Parent=' + obj.parent
    if gff_format == "extended gff3":
        for attribute in _attr_order(obj):
            if type(obj.__dict__[attribute]).__name__ == 'str' and attribute not in _NOT_EXTENDED:
                defline = defline + ';' + attribute + '=' + obj.__dict__[attribute]
    return defline


# ---------------------------------------------------------------------------------------------
# magot_smallfuncs.ensure_file (magot_smallfuncs.py:32-43)
# ---------------------------------------------------------------------------------------------

def ensure_file(potential_file):
    """Path -> opened file, file -> itself, anything unopenable -> the argument as literal text.
    Text is read as latin-1 with '\\n'-only line ends, i.e. byte-for-byte like Python 2."""
    if potential_file is None:
        return None
    if hasattr(potential_file, "read"):
        return potential_file
    try:
        return open(potential_file, encoding="latin-1", newline="\n")
    except (IOError, OSError, ValueError):
        return io.StringIO(potential_file, newline="\n")


def _read_all_bytes(potential_file):
    """ensure_file semantics, returning the whole content as bytes (fast path for big FASTA)."""
    if potential_file is None:
        return None
    if hasattr(potential_file, "read"):
        data = potential_file.read()
        return data.encode("latin-1") if isinstance(data, str) else bytes(data)
    try:
        with open(potential_file, "rb") as fh:
            return fh.read()
    except (IOError, OSError, ValueError, TypeError):
        return potential_file.encode("latin-1") if isinstance(potential_file, str) else bytes(potential_file)


# ---------------------------------------------------------------------------------------------
# Sequence (genome.py:781-851)
# ---------------------------------------------------------------------------------------------

def _device():
    return (DEFAULT_DEVICES or [0])[0]


def _codon_table(library):
    """A caller's codon dict (genome.py:795 `library`) as the 64-byte table of mg_translate_ascii_table.  The reference
    looks up the UPPER-CASED triplet and emits 'X' on a KeyError, so keys that are not upper case or longer than three
    letters can never match and are ignored (1- and 2-letter keys can match the leading fragment of frames 1 and 2, see
    _translate_many); what the device table cannot express is refused: values that are not one byte, and keys that
    contain upper-case symbols other than A, C, G, T (the device path folds all of those into one class)."""
    table = bytearray(b"X" * 64)
    code = {"A": 0, "C": 1, "G": 2, "T": 3}
    for key, value in library.items():
        if not isinstance(key, str) or len(key) != 3 or key != key.upper():
            continue
        if any(ch not in code for ch in key):
            raise NotImplementedError("codon library key %r: only A/C/G/T codons are supported on the device" % (key,))
        if not isinstance(value, str) or len(value.encode("latin-1")) != 1:
            raise NotImplementedError("codon library value %r: only one-byte residues are supported on the device" % (value,))
        table[16 * code[key[0]] + 4 * code[key[1]] + code[key[2]]] = value.encode("latin-1")[0]
    return bytes(table)


def _codon64_of(genetic_code):
    """The 64-byte device table of an NCBI code id, None for the standard code (the default kernels' own table)."""
    code = gencode.check(genetic_code)
    return None if code == 1 else gencode.codon64(code)


_RC_SMALL = {'a': 't', 't': 'a', 'g': 'c', 'c': 'g', 'A': 'T', 'T': 'A', 'G': 'C', 'C': 'G', 'n': 'n', 'N': 'N', '-': '-'}


def _translate_many(seqs, frame=0, strand='+', trimX=True, library=None):
    """Sequence.translate on a batch of byte strings in one launch; returns list of str | None."""
    import ctypes
    n_seq = len(seqs)
    if n_seq == 0:
        return []
    if frame not in (0, 1, 2):
        raise ValueError("frame must be 0, 1 or 2")
    if strand not in ('+', '-'):
        raise UnboundLocalError("local variable 'seq' referenced before assignment")   # genome.py:806-810
    table = None if library is None else _codon_table(library)
    # In frames 1 and 2 the reference first looks up the 1- resp. 2-base fragment before the first full codon
    # (genome.py:811-817, normally a KeyError -> 'X').  A library with such a short key answers it: the device then runs
    # without trimX and the first residue is patched here from the fragment (at most two bases per sequence).
    short_keys = library is not None and frame > 0 and any(isinstance(k, str) and len(k) == frame and k == k.upper() for k in library)
    lens = np.fromiter((len(s) for s in seqs), dtype=np.int64, count=n_seq)
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    data = np.frombuffer(b"".join(seqs), dtype=np.uint8)
    total = int(off[-1])
    cap = (total + 2) // 3 + n_seq + 16
    out = np.empty(cap, dtype=np.uint8)
    out_off = np.zeros(n_seq + 1, dtype=np.int64)
    out_len = np.zeros(n_seq, dtype=np.int64)
    _lib.require_device(_device())
    _lib.check(_lib.lib.mg_translate_ascii_table(_device(), table, ctypes.c_void_p(data.ctypes.data) if total else None,
                                                 ctypes.c_void_p(off.ctypes.data), n_seq, frame, 1 if strand == '-' else 0,
                                                 1 if (trimX and not short_keys) else 0, ctypes.c_void_p(out.ctypes.data), cap,
                                                 ctypes.c_void_p(out_off.ctypes.data), ctypes.c_void_p(out_len.ctypes.data), None))
    buf = out.tobytes()
    res = []
    for i in range(n_seq):
        if out_len[i] < 0:
            res.append(None)
            continue
        r = buf[out_off[i]:out_off[i + 1]].decode("latin-1")
        if short_keys:
            s = seqs[i].decode("latin-1")
            if strand == '-':
                frag = "".join(_RC_SMALL.get(c, 'n') for c in reversed(s[len(s) - 2 * frame:len(s) - frame]))
            else:
                frag = s[frame:2 * frame]
            r = library.get(frag.upper(), 'X') + r[1:]
            if trimX and r[0] == 'X':
                r = r[1:]
        res.append(r)
    return res


class Sequence(str):
    """DNA sequence (genome.py:781).  The work runs on the GPU; results are plain strings."""

    def reverse_compliment(self):
        """genome.py:784-793: reversed, complemented, every byte outside acgtACGTnN- -> 'n'."""
        import ctypes
        n = len(self)
        if n == 0:
            return Sequence("")
        src = np.frombuffer(self.encode("latin-1"), dtype=np.uint8)
        out = np.empty(n, dtype=np.uint8)
        _lib.require_device(_device())
        _lib.check(_lib.lib.mg_revcomp(_device(), ctypes.c_void_p(src.ctypes.data), n, ctypes.c_void_p(out.ctypes.data), None))
        return Sequence(out.tobytes().decode("latin-1"))

    def translate(self, library=None, frame=0, strand='+', trimX=True, genetic_code=1):
        """genome.py:795-822 with the reference's frame quirk; returns None when len <= 2 + frame.
        `library` = a codon -> residue dict (default: the reference's table, NCBI table 1), see _codon_table.
        `genetic_code` = an NCBI table id (magot_b200.gencode); a code other than 1 cannot be combined with `library`."""
        code = gencode.check(genetic_code)
        if code != 1:
            if library is not None:
                raise ValueError("pass either library= or genetic_code=, not both")
            library = gencode.library(code)
        return _translate_many([self.encode("latin-1")], frame=frame, strand=strand, trimX=trimX, library=library)[0]

    def get_orfs(self, longest=False, strand='both', from_atg=False, genetic_code=1):
        """genome.py:824-851 (the `strand` argument is shadowed in the reference and ignored).  `genetic_code`: NCBI table
        id of the translations, and so of the stops the ORFs are split on; start codons stay the reference's 'M' rule."""
        code = gencode.check(genetic_code)
        library = gencode.library(code) if code != 1 else None
        orflist = []
        candidate_list = []
        longest_orf_len = 0
        raw = self.encode("latin-1")
        for frame in (0, 1, 2):
            for st in ('-', '+'):
                translated_seq = _translate_many([raw], frame=frame, strand=st, library=library)[0]
                if translated_seq:
                    for orf in translated_seq.split('*'):
                        output_orf = ('M' + ''.join(orf.split('M')[1:])) if from_atg else orf
                        if longest:
                            if len(output_orf) > longest_orf_len:
                                candidate_list.append(output_orf)
                                longest_orf_len = len(output_orf)
                        else:
                            orflist.append(output_orf)
        if longest:
            return candidate_list[-1]
        return orflist


# ---------------------------------------------------------------------------------------------
# GenomeSequence (genome.py:854-877)
# ---------------------------------------------------------------------------------------------

class DeviceContig(object):
    """Lazy view of one contig held in the packed device genome.  Behaves like the reference's
    plain `str` value for the operations the reference and its tools perform on it (len, slicing,
    concatenation, comparison, iteration); anything else is served by decoding to `str`."""

    __slots__ = ("_gs", "_index", "_len")

    def __init__(self, gs, index, length):
        self._gs = gs
        self._index = index
        self._len = length

    def __len__(self):
        return self._len

    def _fetch(self, lo, hi, minus=False):
        return self._gs._engine().primary.fetch(self._index, lo, hi, minus).decode("latin-1")

    def __str__(self):
        return self._fetch(0, self._len)

    def __repr__(self):
        return repr(str(self))

    def __getitem__(self, key):
        if isinstance(key, slice):
            lo, hi, step = key.indices(self._len)
            if step == 1:
                return self._fetch(lo, hi) if hi > lo else ""
            return str(self)[key]
        i = key + self._len if key < 0 else key
        if not 0 <= i < self._len:
            raise IndexError("string index out of range")
        return self._fetch(i, i + 1)

    def __iter__(self):
        return iter(str(self))

    def __add__(self, other):
        return str(self) + str(other)

    def __radd__(self, other):
        return str(other) + str(self)

    def __eq__(self, other):
        if isinstance(other, (str, DeviceContig)):
            return len(self) == len(other) and str(self) == str(other)
        return NotImplemented

    def __ne__(self, other):
        r = self.__eq__(other)
        return r if r is NotImplemented else not r

    def __hash__(self):
        return hash(str(self))

    def __contains__(self, sub):
        return sub in str(self)

    def __getattr__(self, name):             # any other str method works on the decoded text
        return getattr(str(self), name)


class GenomeSequence(dict):
    """genome sequence class, multi-fasta input (genome.py:854).  Keys are seqids, values are
    `DeviceContig` views; iteration order is the reference's (Python-2.7 dict order)."""

    def __init__(self, genome_sequence=None, truncate_names=False, devices=None):
        dict.__init__(self)
        self._devices = list(devices) if devices is not None else list(DEFAULT_DEVICES or [0])
        self._sharded = None
        self._pending = {}                   # seqid -> np.uint8 array, host text waiting to be packed
        self._index = {}
        data = _read_all_bytes(genome_sequence)
        if data is not None:
            # only the headers are parsed on the host; the record bodies go to the device as they are and K0f drops
            # the line ends there (mg_genome_pack_fasta)
            names, spans = _scan_fasta(data, truncate_names)
            raw = np.frombuffer(data, dtype=np.uint8)
            for name in _order(names):
                self._pending[name] = _RawBody(raw, *spans[name])
                dict.__setitem__(self, name, None)
            self._build()

    # -- packing ------------------------------------------------------------------------------
    def _build(self):
        names = list(dict.keys(self))
        arrays = [self._pending[n] for n in names]
        lens = np.array([a.size for a in arrays], dtype=np.int64)
        if self._sharded is not None:
            self._sharded.close()
        replicas = []
        for dev in self._devices:
            g = engine.DeviceGenome(lens, device=dev)
            for ci, a in enumerate(arrays):
                if isinstance(a, _RawBody):
                    g.pack_fasta(ci, a.raw, a.lo, a.hi)
                else:
                    g.pack(ci, a)
            g.finalize()
            replicas.append(g)
        self._sharded = engine.ShardedGenome(replicas)
        self._index = {}
        for ci, n in enumerate(names):
            self._index[n] = ci
            dict.__setitem__(self, n, DeviceContig(self, ci, int(lens[ci])))
        self._pending = {}
        self._dirty = False

    def _engine(self):
        if self._sharded is None or getattr(self, "_dirty", False):
            self._rebuild_from_values()
        return self._sharded

    def _rebuild_from_values(self):
        pend = {}
        old = self._sharded.primary if self._sharded is not None else None
        for k in dict.keys(self):
            v = dict.__getitem__(self, k)
            if isinstance(v, DeviceContig) and v._gs is self and old is not None:
                # straight from the old replica (str(v) would come back here through _engine() while _dirty is set);
                # _build() closes the old replicas only after every contig has been read
                pend[k] = np.frombuffer(old.fetch(v._index, 0, v._len), dtype=np.uint8)
            else:
                pend[k] = np.frombuffer(str(v).encode("latin-1"), dtype=np.uint8)
        self._pending = pend
        self._build()

    def __setitem__(self, key, value):
        """Assigning a plain string re-packs the genome on next use (rare; the reference allows it)."""
        dict.__setitem__(self, key, value)
        self._dirty = True

    def contig_index(self, seqid):
        self._engine()
        return self._index[seqid]

    def contig_length(self, seqid):
        return len(dict.__getitem__(self, seqid))

    def __getitem__(self, key):
        v = dict.__getitem__(self, key)
        if not isinstance(v, DeviceContig):
            self._engine()
            v = dict.__getitem__(self, key)
        return v

    def close(self):
        if self._sharded is not None:
            self._sharded.close()
            self._sharded = None


class _RawBody(object):
    """Body of one FASTA record as it sits in the file: raw[lo:hi] with line ends, `size` bases without them."""
    __slots__ = ("raw", "lo", "hi", "size")

    def __init__(self, raw, lo, hi, size):
        self.raw, self.lo, self.hi, self.size = raw, lo, hi, size


def _scan_fasta(data, truncate_names):
    """genome.py:856-877 without touching the sequence bytes in Python: header discovery (bytes.find) and, per record, the
    span of its body and its length = body bytes minus CR/LF (counted for all records in one threaded native call,
    mg_count_line_ends).  Empty records are dropped, text before the first header belongs to seqid '', a repeated header
    replaces the earlier record but keeps its place."""
    import ctypes
    n = len(data)
    recs = []                                            # (seqid, body lo, body hi) in file order

    pos = 0 if data[:1] == b">" else data.find(b"\n>")
    if pos < 0:
        recs.append(("", 0, n))
        pos = n
    elif pos > 0 or data[:1] != b">":
        recs.append(("", 0, pos + 1))
        pos += 1
    while pos < n:
        eol = data.find(b"\n", pos)
        if eol < 0:
            eol = n
        raw = data[pos + 1:eol].replace(b"\r", b"").decode("latin-1")
        seqid = raw.split()[0] if truncate_names is True else raw
        nxt = data.find(b"\n>", eol)
        body_hi = n if nxt < 0 else nxt + 1
        recs.append((seqid, min(eol + 1, n), body_hi))
        pos = n if nxt < 0 else nxt + 1
    lo = np.array([r[1] for r in recs], dtype=np.int64)
    hi = np.array([max(r[2], r[1]) for r in recs], dtype=np.int64)
    eols = np.zeros(len(recs), dtype=np.int64)
    if len(recs):
        _lib.check(_lib.lib.mg_count_line_ends(data, n, len(recs), lo.ctypes.data_as(ctypes.c_void_p), hi.ctypes.data_as(ctypes.c_void_p),
                                               eols.ctypes.data_as(ctypes.c_void_p)))
    names = []
    spans = {}
    for (name, a, b), e in zip(recs, eols.tolist()):
        size = (b - a) - e
        if b <= a or size <= 0:
            continue
        if name not in spans:
            names.append(name)
        spans[name] = (a, b, size)
    return names, spans


# ---------------------------------------------------------------------------------------------
# Annotation model (genome.py:524-778)
# ---------------------------------------------------------------------------------------------

class BaseAnnotation(object):
    """Bottom-most level annotation (CDS, match_part, ...), genome.py:586."""

    def __init__(self, ID, seqid, coords, feature_type, parent=None, strand=".", other_attributes={}, annotation_set=None):
        self.ID = ID
        self.seqid = seqid
        self.coords = coords
        self.feature_type = feature_type
        self.annotation_set = annotation_set
        for attribute in other_attributes:
            setattr(self, attribute, other_attributes[attribute])
        self.parent = parent
        self.strand = strand

    def get_coords(self):
        return self.coords

    def get_gff(self, gff_format="simple gff3"):
        """genome.py:616-645 -- one GFF line ("exon added gff3": an exon twin line before every CDS line).
        Returns None without an annotation_set; an unknown format or `gtf` without a parent raise as in the reference
        (UnboundLocalError / TypeError)."""
        if self.annotation_set is None:
            return None
        cols = _gff_columns(self)
        kind = _gff_format_kind(gff_format)
        if kind == "gff3":
            attributes = _gff3_defline(self, gff_format)
        elif kind == "hint":                              # "augustus hint <type> <src> [<pri>]"
            words = gff_format.split()
            cols[2] = words[2]
            attributes = ";pri=".join(["src=" + words[3]] + words[4:5])
        elif kind == "gtf":                               # a parentless feature raises TypeError (str + None), as in the reference
            attributes = 'transcript_id ' + self.parent + ';gene_id ' + self.annotation_set[self.parent].parent
        else:
            raise UnboundLocalError("local variable 'defline' referenced before assignment")
        line = '\t'.join(cols + [attributes])
        if gff_format == "exon added gff3" and cols[2] == "CDS":
            return line.replace('\tCDS\t', '\texon\t').replace('ID=', 'ID=ExonOf') + "\n" + line
        return line

    def get_seq(self):
        """genome.py:603-614: contig[start-1:end] (Python slice clamping), reverse-complemented on '-'.
        Prints and returns None on an invalid strand or any lookup failure, like the reference."""
        try:
            if self.strand == '+' or self.strand == '.' or self.strand == '-':
                gs = self.annotation_set.genome.genome_sequence
                contig = gs[self.seqid]
                lo, hi, _ = slice(self.coords[0] - 1, self.coords[1]).indices(len(contig))
                if hi <= lo:
                    return Sequence("")
                raw = gs._engine().primary.fetch(gs.contig_index(self.seqid), lo, hi, self.strand == '-')
                return Sequence(raw.decode("latin-1"))
            else:
                print(self.ID + ' has invalid strand value "' + self.strand + '"')
        except _lib.MagotError:
            raise
        except Exception:
            print("either base_annotation has not annotation_set, or annotation_set has no genome, or genome has no"
                  "            genome sequence, or genome sequence has no matching seqid, or coords are out of range on that seqid")
            print(self.seqid)


class ParentAnnotation(object):
    """Parent of any BaseAnnotation (genes, transcripts), genome.py:649."""

    def __init__(self, ID, seqid, feature_type, child_list=[], parent=None, strand=".", annotation_set=None, other_attributes={}):
        self.ID = ID
        self.seqid = seqid
        self.feature_type = feature_type
        self.child_list = list(child_list)
        self.parent = parent
        self.annotation_set = annotation_set
        self.strand = strand
        for attribute in other_attributes:
            setattr(self, attribute, other_attributes[attribute])

    def get_coords(self):
        """genome.py:663-675 -- (min, max) over all descendants; None when childless."""
        if len(self.child_list) > 0 and self.annotation_set is not None:
            coords_list = []
            for child in self.child_list:
                child_object = self.annotation_set[child]
                if isinstance(child_object, ParentAnnotation):
                    coords_list = coords_list + list(child_object.get_coords())    # TypeError on None, as the reference
                elif isinstance(child_object, BaseAnnotation):
                    coords_list = coords_list + list(child_object.coords)
            return (min(coords_list), max(coords_list))

    def get_gff(self, gff_format="simple gff3"):
        """genome.py:733-778 -- this feature's line (not for `gtf` / `augustus hint`) followed by its children's,
        children sorted by coordinates (a repeated coordinate pair is keyed (start, end + number of children so
        far)); "exon added gff3" moves every CDS line behind the other lines of the feature."""
        if self.annotation_set is None:
            return None
        cols = _gff_columns(self)                        # evaluated for every format (a childless parent raises here, as its eval does)
        kind = _gff_format_kind(gff_format)
        if kind == "gff3":
            out = ['\t'.join(cols + [_gff3_defline(self, gff_format)])]
        elif kind in ("hint", "gtf"):
            out = []
        else:
            raise UnboundLocalError("local variable 'defline' referenced before assignment")
        by_coords = {}
        for name in self.child_list:
            child = self.annotation_set[name]
            key = child.get_coords()
            if key in by_coords:
                key = (key[0], key[1] + len(by_coords))
            by_coords[key] = child.get_gff(gff_format)
        out.extend(by_coords[key] for key in sorted(by_coords))
        if gff_format == "exon added gff3":
            # the reference removes and re-appends every CDS line while walking a copy of the list: a stable partition
            physical = '\n'.join(out).split('\n')
            is_cds = [ln.split('\t')[2] == "CDS" for ln in physical]
            out = [ln for ln, c in zip(physical, is_cds) if not c] + [ln for ln, c in zip(physical, is_cds) if c]
        return '\n'.join(out)

    def get_fasta(self, seq_type="nucleotide", longest=False, genomic=False, name_from='ID', genetic_code=1):
        """genome.py:677-731.  One device pass for this annotation and all its descendants.  `genetic_code` (NCBI table id)
        translates seq_type="protein"; it changes no length, so longest= picks the same records."""
        codon64 = _codon64_of(genetic_code)
        if genomic is not True and not (len(self.child_list) > 0 and self.annotation_set is not None):
            return ""
        if self.annotation_set is None or self.annotation_set.genome is None:
            return None if genomic is True else ""
        from .flatten import Flattener
        fl = Flattener(self.annotation_set)
        fl.add_top(self, seq_type=seq_type, longest=longest, genomic=genomic, name_from=name_from)
        return fl.run(seq_type, codon64=codon64)


class AnnotationSet(object):
    """A set of annotations of a single genome, one dict per feature type (genome.py:524)."""

    def __init__(self, genome=None):
        self.gene = {}
        self.transcript = {}
        self.CDS = {}
        self.UTR = {}
        self.genome = genome

    def __getattribute__(self, name):
        # A set that read_gff has just made holds the native model only (_PENDING); the tables and objects of the reference's
        # model are built the first time an instance attribute other than `genome` (a table, __dict__) is looked up.
        if _PENDING and (name == "__dict__" or (name not in _ASET_CLASS_NAMES and name != "genome")) and self in _PENDING:
            _materialise(self)
        return object.__getattribute__(self, name)

    def _dict_names(self):
        return sorted(k for k, v in self.__dict__.items() if type(v) == dict)

    def __getitem__(self, item):
        """genome.py:536-544: look in every dict attribute in dir() (sorted) order; the LAST hit wins."""
        hit = None
        found = False
        d = self.__dict__
        for name in self._dict_names():
            t = d[name]
            try:
                hit = t[item]
                found = True
            except (KeyError, TypeError):
                pass
        if not found:
            raise KeyError(item)
        return hit

    def build_index(self):
        """ID -> object for every feature with __getitem__'s precedence (one pass, used by the flattener).  Kept between calls
        (module-level weak map, so the set's __dict__ stays the reference's) and rebuilt when a table has been added, removed,
        replaced or has changed size -- the loop `for t in aset.transcript.values(): t.get_fasta()` costs one pass, not one
        per call.  Bulk extraction should still go through AnnotationSet.get_fasta (one device plan for all records)."""
        d = self.__dict__
        names = self._dict_names()
        stamp = tuple((name, id(d[name]), len(d[name])) for name in names)
        hit = _INDEX_CACHE.get(self)
        if hit is not None and hit[0] == stamp:
            return hit[1]
        idx = {}
        for name in names:
            idx.update(d[name])
        _INDEX_CACHE[self] = (stamp, idx)
        return idx

    def get_seqid(self, seqid):
        """genome.py:550-559 -- a new AnnotationSet holding the features that sit on `seqid` (same objects), one table
        per table of this set; features are filed under their own feature_type."""
        seqid_annotation_set = AnnotationSet()
        for name in self._dict_names():
            setattr(seqid_annotation_set, name, {})
            for feature, feature_obj in self.__dict__[name].items():
                if feature_obj.seqid == seqid:
                    getattr(seqid_annotation_set, feature_obj.feature_type)[feature] = feature_obj
        for name in seqid_annotation_set._dict_names():
            tbl = seqid_annotation_set.__dict__[name]
            seqid_annotation_set.__dict__[name] = {k: tbl[k] for k in _order(list(tbl))}
        return seqid_annotation_set

    def get_all_seqids(self):
        """genome.py:561-567 -- list(set(...)) of every feature's seqid, in the order a Python-2.7 set iterates
        (same table discipline as the 2.7 dict: setobject.c set_add_entry / set_table_resize)."""
        seen = {}
        for name in self._dict_names():
            for feature_obj in self.__dict__[name].values():
                seen.setdefault(feature_obj.seqid, None)
        return _order(list(seen))

    def read_gff(self, gff, *args, **kwargs):
        kwargs["annotation_set_to_modify"] = self
        read_gff(gff, *args, **kwargs)

    def read_cegma_gff(self, cegma_gff):
        read_cegma_gff(cegma_gff, annotation_set_to_modify=self)

    def read_exonerate(self, exonerate_output):
        read_exonerate(exonerate_output, annotation_set_to_modify=self)

    def read_blast_csv(self, blast_csv, hierarchy=['match', 'match_part'], source='blast', find_truncated_locname=False):
        read_blast_csv(blast_csv, annotation_set_to_modify=self, hierarchy=hierarchy, source=source,
                       find_truncated_locname=find_truncated_locname)

    def get_fasta(self, feature, seq_type="nucleotide", longest=False, genomic=False, genetic_code=1):
        """genome.py:578-582: '\\n'.join of every <feature> annotation's fasta, in dict order
        (empty results stay in the list -> blank lines).  All records go through ONE device plan.  A set that still holds
        the native model of its read_gff call is flattened there (no Python object per feature).  `genetic_code` (NCBI
        table id) translates seq_type="protein"."""
        codon64 = _codon64_of(genetic_code)
        model = _PENDING.get(self) if _PENDING else None
        if model is not None:
            text = _native_get_fasta(self, model, feature, seq_type, longest, genomic, codon64)
            if text is not None:
                return text
        table = getattr(self, feature)
        from .flatten import Flattener
        fl = Flattener(self)
        for key in table:
            obj = table[key]
            if not hasattr(obj, "get_fasta"):
                raise AttributeError("%s instance has no attribute 'get_fasta'" % obj.__class__.__name__)
            fl.add_top(obj, seq_type=seq_type, longest=longest, genomic=genomic, name_from='ID')
        return fl.run(seq_type, codon64=codon64)


    def check_cds(self, feature, genetic_code=1, start_codons=("ATG",), use_phase=False, codon_usage=True, junctions=True):
        """Gene-model check (mg_plan_check) of exactly the records get_fasta(feature, seq_type="protein") prints, in its
        order: start / stop codons, in-frame stops, reading frame, ambiguous codons, GC, splice sites and codon usage under
        NCBI table `genetic_code`.  start_codons: codons a CDS may start with; use_phase: start at the GFF phase of the first
        CDS.  Returns CdsCheck(names, records (engine.CHECK_DTYPE), codon_counts (uint32 [n, 64] or None), junctions (int8
        class after each segment, or None), seg_off (segments of record i: junctions[seg_off[i]:seg_off[i+1]])).  The names
        are the records' FASTA headers without '>'."""
        code = gencode.check(genetic_code)
        starts = gencode.start64(start_codons, code)      # ValueError before any device work
        gs, tbl = _feature_table(self, feature, "protein")
        if tbl is None or tbl.n_rec == 0:
            return CdsCheck([], np.zeros(0, dtype=engine.CHECK_DTYPE), np.zeros((0, 64), np.uint32) if codon_usage else None,
                            np.zeros(0, np.int8) if junctions else None, np.zeros(1, np.int64))
        plan = engine.Plan(gs._engine().primary, tbl)
        try:
            if code != 1:
                plan.set_codon_table(gencode.codon64(code))
            plan.prepare_async(trimx=False, defer_records=True)     # the check needs the piece pass only
            recs, counts, junc = plan.check(starts, use_phase=use_phase, codon_usage=codon_usage, junctions=junctions)
        finally:
            plan.close()
        keep = np.flatnonzero(tbl.rec_pre_len > 0)        # FASTA records; the blank entries of empty tops have no header
        names = _record_names(tbl, keep)
        nseg = np.diff(tbl.rec_seg_off)[keep]
        seg_off = np.concatenate(([0], np.cumsum(nseg))).astype(np.int64)
        if junc is not None:
            rows = np.concatenate([np.arange(tbl.rec_seg_off[r], tbl.rec_seg_off[r + 1]) for r in keep.tolist()]) if keep.size else np.zeros(0, np.int64)
            junc = junc[rows.astype(np.int64)]
        return CdsCheck(names, recs[keep], counts[keep] if counts is not None else None, junc, seg_off)

    def predict_cds(self, feature="gene", min_aa=100, genetic_code=1, start_codons=("ATG",), partial5=False, partial3=False,
                    strand="sense"):
        """CDS prediction (mg_plan_predict_cds) for exactly the records get_fasta(feature, seq_type="nucleotide") prints, in its
        order, e.g. exon-only transcript models: the longest ORF of each spliced transcript in its three frames, at least
        min_aa residues, from a codon in start_codons to a stop of NCBI table `genetic_code`; partial5 / partial3 also accept
        ORFs open at the 5' end of a frame / without a stop.  strand="both" also scores the antisense (the reverse complement of
        the transcript): per record the longer ORF wins, the sense one on a tie.  Returns CdsPrediction(names, records
        (engine.PRED_DTYPE, coordinates in the chosen strand's transcript), antisense (int8, 1 where the antisense ORF was
        chosen), seg_contig, seg_lo, seg_hi (0-based half-open forward coordinates), seg_strand (0 '+', 1 '-'), seg_phase: the
        CDS segments of record i in transcript order are seg_*[seg_off[i]:seg_off[i+1]], none for a record without an ORF)."""
        code = gencode.check(genetic_code)
        starts = gencode.start64(start_codons, code)      # ValueError before any device work
        if strand not in ("sense", "both"):
            raise ValueError("strand %r is not 'sense' or 'both'" % (strand,))
        if isinstance(min_aa, bool) or int(min_aa) != min_aa or int(min_aa) < 0:
            raise ValueError("min_aa %r is not a count of residues" % (min_aa,))
        gs, tbl = _feature_table(self, feature, "nucleotide")
        if tbl is None or tbl.n_rec == 0:
            return _empty_prediction()
        flags = dict(min_aa=int(min_aa), start_codons=starts, partial5=bool(partial5), partial3=bool(partial3))
        recs, segs = _predict_table(gs, tbl, code, **flags)
        contig, seg_strand = tbl.seg_contig, tbl.seg_strand
        anti = np.zeros(tbl.n_rec, dtype=np.int8)
        if strand == "both":
            at = antisense_table(tbl)
            recs2, segs2 = _predict_table(gs, at, code, **flags)
            anti = (recs2["n_aa"] > recs["n_aa"]).astype(np.int8)
            rep = np.repeat(anti, np.diff(tbl.rec_seg_off)).astype(bool)
            recs = np.where(anti.astype(bool), recs2, recs)
            segs = np.where(rep, segs2, segs)
            contig = np.where(rep, at.seg_contig, tbl.seg_contig)
            seg_strand = np.where(rep, at.seg_strand, tbl.seg_strand)
        keep = np.flatnonzero(tbl.rec_pre_len > 0)        # FASTA records; the blank entries of empty tops have no header
        keep_seg = np.repeat(tbl.rec_pre_len > 0, np.diff(tbl.rec_seg_off)) & (segs["lo"] >= 0)
        seg_off = np.concatenate(([0], np.cumsum(recs["n_cds_seg"][keep]))).astype(np.int64)
        return CdsPrediction(_record_names(tbl, keep), recs[keep], anti[keep], contig[keep_seg].astype(np.int32),
                             segs["lo"][keep_seg], segs["hi"][keep_seg], seg_strand[keep_seg].astype(np.int8),
                             segs["phase"][keep_seg], seg_off)


CdsCheck = collections.namedtuple("CdsCheck", "names records codon_counts junctions seg_off")
CdsPrediction = collections.namedtuple("CdsPrediction", "names records antisense seg_contig seg_lo seg_hi seg_strand seg_phase "
                                                        "seg_off")


def _empty_prediction():
    z = np.zeros(0, np.int64)
    return CdsPrediction([], np.zeros(0, dtype=engine.PRED_DTYPE), np.zeros(0, np.int8), np.zeros(0, np.int32), z, z,
                         np.zeros(0, np.int8), np.zeros(0, np.int8), np.zeros(1, np.int64))


def _feature_table(annotation_set, feature, seq_type):
    """(genome sequence, RecordTable) of what annotation_set.get_fasta(feature, seq_type) prints: the native model's table
    when the set still holds one, else the Flattener's; the table is None without records."""
    model = _PENDING.get(annotation_set) if _PENDING else None
    flat = _native_table(annotation_set, model, feature) if model is not None else None
    if flat is not None:
        return flat[0], flat[1]
    table = getattr(annotation_set, feature)
    from .flatten import Flattener
    fl = Flattener(annotation_set)
    for key in table:
        obj = table[key]
        if not hasattr(obj, "get_fasta"):
            raise AttributeError("%s instance has no attribute 'get_fasta'" % obj.__class__.__name__)
        fl.add_top(obj, seq_type=seq_type, longest=False, genomic=False, name_from='ID')
    return fl.gs, fl.records(seq_type)[0]


def _record_names(tbl, rows):
    """FASTA headers without '>' of the records `rows` of a framed table."""
    lit = tbl.lit.tobytes()
    return [lit[o + 1:o + n - 1].decode("latin-1") for o, n in zip(tbl.rec_lit_off[rows].tolist(), tbl.rec_pre_len[rows].tolist())]


def antisense_table(tbl):
    """The table whose record r is the reverse complement of record r of tbl: its segments in reverse order, strands flipped
    (literals and phases kept)."""
    cnt = np.diff(tbl.rec_seg_off)
    rep = np.repeat(np.arange(tbl.n_rec), cnt)
    idx = tbl.rec_seg_off[rep + 1] - 1 - (np.arange(tbl.n_seg) - tbl.rec_seg_off[rep])
    return engine.RecordTable(tbl.rec_seg_off, tbl.seg_contig[idx], tbl.seg_start[idx], tbl.seg_end[idx], tbl.seg_strand[idx] == 0,
                              tbl.rec_lit_off, tbl.rec_pre_len, tbl.rec_suf_len, tbl.lit, tbl.rec_phase)


def _predict_table(gs, tbl, code, min_aa, start_codons, partial5, partial3):
    plan = engine.Plan(gs._engine().primary, tbl)
    try:
        if code != 1:
            plan.set_codon_table(gencode.codon64(code))
        plan.prepare_async(trimx=False, defer_records=True)     # the prediction needs the piece pass only
        return plan.predict_cds(min_aa, start_codons, partial5, partial3)
    finally:
        plan.close()

_ASET_CLASS_NAMES = frozenset(dir(AnnotationSet))


def _materialise(annotation_set):
    """Native model -> the reference's tables and objects (once; the set stops being 'pending')."""
    model = _PENDING.pop(annotation_set, None)
    if model is None:
        return
    import gc
    was_enabled = gc.isenabled()
    gc.disable()                                         # millions of long-lived objects: generation-2 passes walk them for nothing
    try:
        _apply_model(annotation_set, object.__getattribute__(annotation_set, "__dict__"), model, [], deepcopy_order=True)
    finally:
        if was_enabled:
            gc.enable()
    model.close()


def _native_get_fasta(annotation_set, model, feature, seq_type, longest, genomic, codon64=None):
    """AnnotationSet.get_fasta on the native model: tops in the set's (Python-2.7 dict, after deepcopy) order, children chosen
    and ordered by mg_gff_flatten, one device plan.  Returns None when the call needs the object model (genomic spans,
    longest=, an unknown table, a model the flattener refuses: the object path then prints / raises like the reference)."""
    if genomic is True or longest is True or seq_type not in ("nucleotide", "protein") or not isinstance(feature, str):
        return None
    import time as _time
    t0 = _time.perf_counter()
    flat = _native_table(annotation_set, model, feature)
    if flat is None:
        return None
    gs, tbl, rec_name = flat
    protein = seq_type == "protein"
    t1 = _time.perf_counter()
    text, lens = gs._engine().run_table(tbl, protein=protein, want_lengths=protein, codon64=codon64)
    t2 = _time.perf_counter()
    if protein and lens is not None and ((lens[1] < 0) & (rec_name >= 0)).any():
        # Sequence.translate returned None (spliced length <= 2): '>' + name + '\n' + None (genome.py:710)
        raise TypeError("cannot concatenate 'str' and 'NoneType' objects")
    out = engine.decode_text(text, strip_last=1)
    if TIMINGS is not None:
        TIMINGS.update({"flatten_s": t1 - t0, "device_and_copy_s": t2 - t1, "decode_s": _time.perf_counter() - t2,
                        "records": int(tbl.n_rec), "segments": int(tbl.n_seg), "text_bytes": len(text)})
    return out


def _native_table(annotation_set, model, feature):
    """(genome sequence, RecordTable, rec_name ids) of AnnotationSet.get_fasta(feature) on the native model, framed as the
    FASTA text; None when the call needs the object model."""
    genome = object.__getattribute__(annotation_set, "__dict__").get("genome")
    gs = getattr(genome, "genome_sequence", None) if genome is not None else None
    if gs is None:
        return None
    rows = model.table_rows(feature)
    if rows is None or rows.size == 0:
        return None
    ids = model.column("id")[rows]
    if np.unique(ids).size != ids.size:                  # interned: equal strings <=> equal ids
        return None
    # tops in the order the reference's table dict iterates after its deepcopy, computed on the model's strings
    tops = np.ascontiguousarray(rows[model.py2_order(ids, deepcopy=True)] if RECORD_ORDER == "py2" else rows, dtype=np.int64)
    seq_ids = np.unique(model.column("seqid"))
    seq_ids = seq_ids[seq_ids >= 0]
    contig_of = np.full(model.n_strings, -1, dtype=np.int32)
    for sid, name in zip(seq_ids.tolist(), model.strings(seq_ids)):
        if dict.__contains__(gs, name):
            contig_of[sid] = gs.contig_index(name)
    tbl, top_rec_off, rec_name = model.flatten(tops, contig_of, framing=True)
    if tbl is None:
        return None
    return gs, tbl, rec_name


def write_gff(annotation_set, gff_format="simple gff3"):
    """genome.py:228-238 -- GFF text of every feature table whose first entry has no parent, tables taken in the
    iteration order of the set's instance dict, features in table (Python-2.7 dict) order."""
    gff_lines = []
    adict = annotation_set.__dict__
    for attribute in _attr_order(annotation_set):
        table = adict[attribute]
        if type(table) == dict and len(table) > 0:
            first = table[next(iter(table))]
            if first.__class__.__name__ in ("ParentAnnotation", "BaseAnnotation") and first.parent is None:
                for annotationID in table:
                    gff_lines.append(table[annotationID].get_gff(gff_format))
    return '\n'.join(gff_lines)


_AUGUSTUS_IGNORE = ['gene', 'transcript', 'stop_codon', 'terminal', 'internal', 'initial', 'intron', 'start_codon', 'single']


def read_gff(gff, annotation_set_to_modify=None, base_features=['CDS', 'match_part', 'similarity', 'region'],
             features_to_ignore=['exon'], gff_version="auto", parents_hierarchy=[], features_to_replace=[],
             IDfield="ID", parent_field="Parent", presets=None):
    """genome.py:242-415 -- GFF3 / GTF reader with the reference's ID, de-dup and implicit-parent semantics.

    The text is tokenised and interpreted by the native reader (csrc/mg_gff.cu through magot_b200.gffnative): lines become
    rows of interned integer ids, IDs are named / de-duplicated and parents created on those ids.  Without
    annotation_set_to_modify a new AnnotationSet is returned that HOLDS that model: `get_fasta(feature)` flattens it straight
    into interval tables for the device, and the reference's Python objects (dicts in the order the reference's deepcopy
    leaves them, genome.py:415) are built only when a table, an object or the set's __dict__ is touched.  With
    annotation_set_to_modify the rows are added to that set's objects right away."""
    from . import gffnative
    # presets (genome.py:261-268): the reference exec()s these assignments, which rebinds the locals under Python 2;
    # a name that is not a preset (e.g. convert_gff's input_format 'gtf') changes nothing.
    if presets == "augustus":
        features_to_ignore = list(_AUGUSTUS_IGNORE)
        parent_field = None
        parents_hierarchy = ['transcript_id', 'gene_id']
        IDfield = None
    elif presets == "RepeatMasker":
        parent_field = None
        IDfield = 'Target'
    elif presets == "CEGMA":
        # the preset text indexes a list literal with a tuple ([['First','CDS']['Internal','CDS']...]): the exec raises
        raise TypeError("list indices must be integers, not tuple")
    text = _read_all_bytes(gff)                        # ensure_file semantics (path, file object or literal text), as bytes
    version = 0 if gff_version == "auto" else (gff_version if gff_version in (2, 3) and not isinstance(gff_version, bool) else -1)
    fresh = annotation_set_to_modify is None
    table_names, nondict, existing, ext_objects = [], [], [], []
    if fresh:
        annotation_set = AnnotationSet()
        adict = object.__getattribute__(annotation_set, "__dict__")
    else:
        annotation_set = annotation_set_to_modify
        adict = annotation_set.__dict__                 # (materialises a set that still holds a native model)
    for name, v in adict.items():
        if type(v) == dict:
            table_names.append(name)
        else:
            nondict.append(name)
    if not fresh:
        for t, name in enumerate(table_names):
            for ID, obj in adict[name].items():
                if isinstance(ID, str):
                    kids = getattr(obj, "child_list", None)
                    existing.append((t, ID, isinstance(kids, list), [c for c in kids if isinstance(c, str)] if isinstance(kids, list) else []))
                    ext_objects.append(obj)
    # whole-line replacement of "\tX\t" by "\tY\t" (genome.py:271-272)
    replace = [("\t" + f[0] + "\t", "\t" + f[1] + "\t") for f in features_to_replace]
    opts = gffnative.pack_opts(version, features_to_ignore, base_features, list(parents_hierarchy), replace,
                               IDfield, parent_field, table_names, nondict, existing)
    model = gffnative.Model(text, opts)
    st = model.status
    if fresh and st == gffnative.STATUS_OK:
        _PENDING[annotation_set] = model
        return annotation_set
    if not fresh or st not in (gffnative.GFF2_NO_VALUE, gffnative.MISSING_PARENT):
        _apply_model(annotation_set, adict, model, ext_objects, deepcopy_order=False)
    if st == gffnative.STATUS_OK:
        return None
    if st == gffnative.GFF2_NO_VALUE:
        print(model.string(model.err_a))
        return None
    if st == gffnative.MISSING_PARENT:
        print("""It seems that this line has a parent attribute but that that parent doesn't have a line itself nor
                    does this line have a defline attribute that specifies a parent type. I'm afraid this function can't currently
                    deal with that.""")
        print(model.string(model.err_a))
        print(model.string(model.err_b))
        return None
    if st == gffnative.BAD_INT:
        raise ValueError("invalid literal for int() with base 10: %r" % model.string(model.err_a))
    if st == gffnative.PARENT_IS_BASE:
        raise AttributeError("'BaseAnnotation' object has no attribute 'child_list'")
    if st == gffnative.ATTR_CLASH:
        raise TypeError("'%s' object does not support item assignment" % type(adict.get(model.string(model.err_a))).__name__)
    if st == gffnative.NONE_TWICE:
        raise TypeError("unsupported operand type(s) for +: 'NoneType' and 'str'")
    raise IndexError("list index out of range")


# AnnotationSets that still hold the native model of the read_gff call that made them (no Python object built yet)
_PENDING = weakref.WeakKeyDictionary()
_INDEX_CACHE = weakref.WeakKeyDictionary()              # AnnotationSet -> (stamp of its tables, ID -> object)


def _apply_model(annotation_set, adict, model, ext_objects, deepcopy_order):
    """Build the reference's objects from a native model: one BaseAnnotation / ParentAnnotation per row through the same
    constructors (so attribute precedence is the reference's), tables filled in dict insertion order; rows that stand
    for objects the set already had only receive their new children."""
    S = model.all_strings()
    n = model.n_rows
    col = model.column
    ids, seqid, ftype, strand, source, parent = (col(k).tolist() for k in ("id", "seqid", "ftype", "strand", "source", "parent"))
    start, end, score, has_score, phase = (col(k).tolist() for k in ("start", "end", "score", "has_score", "phase"))
    is_base, implicit, ext, attr0, nattr = (col(k).tolist() for k in ("is_base", "implicit", "ext", "attr0", "nattr"))
    child_off, child, ext0 = col("child_off").tolist(), col("child").tolist(), col("ext_children0").tolist()
    akey, aval = col("attr_key").tolist(), col("attr_val").tolist()
    objs = [None] * n
    for r in range(n):
        kids = [S[c] for c in child[child_off[r]:child_off[r + 1]]]
        if ext[r] >= 0:
            obj = ext_objects[ext[r]]
            if isinstance(getattr(obj, "child_list", None), list):
                obj.child_list.extend(kids[ext0[r]:])
            objs[r] = obj
            continue
        par = S[parent[r]] if parent[r] >= 0 else None
        if implicit[r]:
            objs[r] = ParentAnnotation(S[ids[r]], S[seqid[r]], S[ftype[r]], child_list=kids, parent=par, strand=S[strand[r]],
                                       annotation_set=annotation_set)
            continue
        other = {'source': S[source[r]]}
        if has_score[r]:
            other['score'] = score[r]
        if phase[r] >= 0:
            other['phase'] = phase[r]
        a0 = attr0[r]
        for k in range(a0, a0 + nattr[r]):
            other[S[akey[k]]] = S[aval[k]]
        if is_base[r]:
            objs[r] = BaseAnnotation(S[ids[r]], S[seqid[r]], (start[r], end[r]), S[ftype[r]], par, S[strand[r]], other, annotation_set)
        else:
            obj = ParentAnnotation(S[ids[r]], S[seqid[r]], S[ftype[r]], [], par, S[strand[r]], annotation_set, other)
            if 'child_list' not in other:
                obj.child_list = kids
            objs[r] = obj
    tname, toff, trows = col("table_name").tolist(), col("table_off").tolist(), col("table_rows").tolist()
    for t, name_id in enumerate(tname):
        name = S[name_id]
        if name not in adict:
            adict[name] = {}
        tbl = adict[name]
        for r in trows[toff[t]:toff[t + 1]]:
            if ext[r] < 0:
                tbl[S[ids[r]]] = objs[r]
    if deepcopy_order:
        # copy.deepcopy (genome.py:415) re-inserts every dict in Python-2.7 slot order
        for name in sorted(k for k, v in adict.items() if type(v) == dict):
            tbl = adict[name]
            if tbl:
                adict[name] = {k: tbl[k] for k in _order(list(tbl), deepcopy=True)}
        _DEEPCOPIED_SETS.add(annotation_set)


def read_cegma_gff(cegma_gff, annotation_set_to_modify=None):
    """genome.py:418-422.  The reference's CEGMA preset text is malformed, so this raises TypeError there and here."""
    annotation_set = read_gff(cegma_gff, annotation_set_to_modify=annotation_set_to_modify, presets="CEGMA")
    if annotation_set_to_modify is None:
        return annotation_set


def _py2_reorder(annotation_set):
    """Leave every feature dict in the order a CPython-2.7 dict would iterate after these insertions (no deepcopy on
    the read_blast_csv / read_exonerate paths: both fill the set they are given, genome.py:88-120, :425-499)."""
    adict = annotation_set.__dict__
    for name in annotation_set._dict_names():
        tbl = adict[name]
        if tbl:
            adict[name] = {k: tbl[k] for k in _order(list(tbl), deepcopy=False)}


def vulgar2gff(vulgarlist, feature_types=['match', 'match_part'], source='exonerate'):
    """genome.py:32-85 -- one exonerate `vulgar:` line (already split) -> GFF3 lines: a top-level hit and one
    sub-feature per run of M/S/G/F triples.  Quirk kept: the sub-feature's coordinates are the min/max of the
    positions AS STRINGS (lexicographic), as the reference computes them."""
    qname = vulgarlist[0] + '-against-' + vulgarlist[4]
    tname, tstart, tend, tstrand, score = vulgarlist[4], vulgarlist[5], vulgarlist[6], vulgarlist[7], vulgarlist[8]
    triples = vulgarlist[9:]
    if tstrand == "+":
        tposition = int(tstart) + 1
    else:
        tposition = int(tstart)
        tend = str(int(tend) + 1)
    gfflines = ["\t".join([tname, source, feature_types[0], str(tposition), tend, score, tstrand, '.', 'ID=' + qname])]
    open_feature = False
    coords = []
    IDnum = 1

    def close():
        return '\t'.join([tname, source, feature_types[1], str(min(coords)), str(max(coords)), '.', tstrand, '.',
                          'ID=' + qname + '_' + feature_types[1] + str(IDnum) + ';Parent=' + qname])

    for i, field in enumerate(triples):
        if i % 3 == 0:
            if field in ('M', 'S', 'G', 'F'):
                if not open_feature:
                    open_feature = True
                    coords = [str(tposition)]
            elif open_feature:
                gfflines.append(close())
                IDnum += 1
                open_feature = False
        if i % 3 == 2:
            if tstrand == "+":
                tposition += int(field)
            elif tstrand == "-":
                tposition -= int(field)
            if open_feature:
                if tstrand == '+':
                    coords.append(str(tposition - 1))
                elif tstrand == '-':
                    coords.append(str(tposition + 1))
    if open_feature:
        gfflines.append(close())
    return '\n'.join(gfflines)


def read_exonerate(exonerate_output, annotation_set_to_modify=None):
    """genome.py:88-120 -- exonerate text output (Query:/Target:/vulgar: lines) -> match / match_part annotations."""
    annotation_set = AnnotationSet() if annotation_set_to_modify is None else annotation_set_to_modify
    gfflines = []
    seen = {}
    qname = ""
    tname = ""
    for original_line in ensure_file(exonerate_output):
        line = original_line.replace('\r', '').replace('\n', '')
        if line[:16] == "         Query: ":
            qname = line[16:]
        elif line[:16] == "        Target: ":
            tname = line[16:].replace(':[revcomp]', '').replace('[revcomp]', '')
            if tname[-1] == " ":
                tname = tname[:-1]
        elif line[:8] == "vulgar: ":
            v = line[8:].split()
            v[0] = qname                              # names with spaces survive: the header lines win over the vulgar fields
            v[4] = tname
            ID = v[0] + '-against-' + v[4]
            if ID in seen:
                v[0] = v[0] + str(seen[ID])
                seen[ID] += 1
            else:
                seen[ID] = 1
            gfflines.append(vulgar2gff(v))
    read_gff("\n".join(gfflines), annotation_set_to_modify=annotation_set)
    _py2_reorder(annotation_set)
    if annotation_set_to_modify is None:
        return annotation_set


def read_blast_csv(blast_csv, annotation_set_to_modify=None, hierarchy=['match', 'match_part'], source='blast',
                   find_truncated_locname=False):
    """genome.py:425-499 -- blast -outfmt 10 lines -> one base feature per hit plus its chain of single-child parents.
    Hits are not strung together; repeated query IDs become ID-1, ID-2, ..."""
    blast_file = ensure_file(blast_csv)
    annotation_set = AnnotationSet() if annotation_set_to_modify is None else annotation_set_to_modify
    adict = annotation_set.__dict__
    next_suffix = {}
    feature_type = hierarchy[-1]
    parents_chain = list(hierarchy[:-1])
    parents_chain.reverse()
    if feature_type not in adict:
        adict[feature_type] = {}
    genome_seqids = None
    if find_truncated_locname:
        if annotation_set.genome is None:
            print('"warning: find_truncated_locname" was set to true, but annotation set has no associated genome object so this '
                  'cannot be done')
            find_truncated_locname = False
        else:
            genome_seqids = annotation_set.genome.get_seqids()
    for whole_line in blast_file:
        fields = whole_line.replace('\r', '').replace('\n', '').split(',')
        if len(fields) <= 8:
            continue
        seqid = fields[1]
        if find_truncated_locname and seqid not in genome_seqids:
            for genome_seqid in genome_seqids:
                if seqid == genome_seqid.split()[0]:
                    seqid = genome_seqid
                    break
        tstart, tend = int(fields[8]), int(fields[9])
        if tstart < tend:
            coords, strand = (tstart, tend), '+'
        else:
            coords, strand = (tend, tstart), '-'
        IDbase = fields[0]
        base_tbl = adict[feature_type]
        if IDbase in base_tbl:
            ID = IDbase + '-' + str(next_suffix[IDbase])
            next_suffix[IDbase] += 1
            while ID in base_tbl:
                ID = IDbase + '-' + str(next_suffix[IDbase])
                next_suffix[IDbase] += 1
        else:
            ID = IDbase
            next_suffix[IDbase] = 1
        other_attributes = {'evalue': fields[10], 'score': fields[11]}
        parent = ID + '-' + parents_chain[0]
        child_to_set = ID
        for k, parent_feature in enumerate(parents_chain):
            if parent_feature not in adict:
                adict[parent_feature] = {}
            parent_to_set = ID + '-' + parents_chain[k + 1] if k != len(parents_chain) - 1 else None
            adict[parent_feature][ID + '-' + parent_feature] = ParentAnnotation(
                ID + '-' + parent_feature, seqid, parent_feature, [child_to_set], parent_to_set, strand, annotation_set,
                other_attributes={})
            child_to_set = ID + '-' + parent_feature
        base_tbl[ID] = BaseAnnotation(ID, seqid, coords, feature_type, parent, strand, other_attributes, annotation_set)
    _py2_reorder(annotation_set)
    if annotation_set_to_modify is None:
        return annotation_set

# ---------------------------------------------------------------------------------------------
# position_dic (genome.py:981-1100): per-base arrays; AT content and window sums run on the device (K6)
# ---------------------------------------------------------------------------------------------

class position_dic(dict):
    """seqid -> numpy array with one element per base (genome.py:981).  The arrays live on the host, as in the reference
    (callers index and assign them directly); `at_content` reads the packed genome on the device and
    `sliding_window_calculate` sums windows through a device prefix scan instead of one numpy.sum per window."""

    def __init__(self, genome_sequence, dtype=bool):
        seqids = list(genome_sequence)
        for seqid in _order(seqids):                 # a position_dic is a Python-2.7 dict itself: its own slot order
            self[seqid] = np.zeros(len(genome_sequence[seqid]), dtype=dtype)

    @staticmethod
    def _positions(arr, coords):
        """Index array of `for position in range(coords[0] - 1, coords[1])` on a numpy array, up to the first position
        numpy would refuse (negative positions wrap like numpy's), and that position (or None)."""
        n = len(arr)
        lo, hi = coords[0] - 1, coords[1]
        bad = None
        if lo < -n:
            bad, hi = lo, lo
        elif hi > n:
            bad, hi = max(n, lo), max(n, lo)
        return np.arange(lo, max(hi, lo)), bad, n

    def fill_from_annotations(self, annotation_set, feature, fill_type="coords", fill_with="1"):
        """genome.py:986-1004.  accepts "start" and "coords" for fill_type; fill_with is evaluated like the reference's
        eval(), once per annotation unless it mentions `position`."""
        table = getattr(annotation_set, feature)
        for annotation in table:
            annotation_obj = table[annotation]
            seqid = annotation_obj.seqid
            coords = annotation_obj.get_coords()
            try:
                parent = annotation_obj.parent
            except Exception:
                parent = None
            ID = annotation_obj.ID
            scope = dict(globals())
            scope.update(self=self, annotation_set=annotation_set, feature=feature, fill_type=fill_type, fill_with=fill_with,
                         annotation=annotation, annotation_obj=annotation_obj, seqid=seqid, coords=coords, parent=parent, ID=ID,
                         numpy=np)
            if fill_type == "coords":
                arr = self[seqid]
                idx, bad, n = self._positions(arr, coords)
                if "position" in fill_with:
                    for position in idx.tolist():
                        scope["position"] = position
                        arr[position] = eval(fill_with, scope)
                elif idx.size:
                    arr[idx] = eval(fill_with, scope)
                if bad is not None:
                    raise IndexError("index %d is out of bounds for axis 0 with size %d" % (bad, n))
            elif fill_type == "start":
                scope["position"] = None
                self[seqid][coords[0] - 1] = eval(fill_with, scope)

    def count_from_annotations(self, annotation_set, feature):
        """genome.py:1006-1027 -- [featureID, positions equal to 0, positions equal to 1] per annotation."""
        count_list = []
        table = getattr(annotation_set, feature)
        for annotation in table:
            annotation_obj = table[annotation]
            arr = self[annotation_obj.seqid]
            idx, bad, n = self._positions(arr, annotation_obj.get_coords())
            if bad is not None:
                raise IndexError("index %d is out of bounds for axis 0 with size %d" % (bad, n))
            vals = arr[idx]
            count_list.append([annotation_obj.ID, int(np.count_nonzero(vals == 0)), int(np.count_nonzero(vals == 1))])
        return count_list

    def at_content(self, genome_sequence):
        """genome.py:1030-1034 -- set position to 1 wherever the base is one of "ATat" (nothing is cleared)."""
        import ctypes
        gs = genome_sequence
        if not isinstance(gs, GenomeSequence):
            gs = GenomeSequence()
            for k in genome_sequence:
                gs[k] = genome_sequence[k]
        for seqid in self:
            arr = self[seqid]
            L = len(gs[seqid])
            m = min(len(arr), L)
            if m:
                flags = np.empty(m, dtype=np.uint8)
                eng = gs._engine().primary
                _lib.check(_lib.lib.mg_genome_at_flags(eng.handle, gs.contig_index(seqid), 0, m, ctypes.c_void_p(flags.ctypes.data), None))
                arr[:m][flags != 0] = 1
            if len(arr) > L:
                raise IndexError("string index out of range")

    @staticmethod
    def _window_sums(arr, window_size, window_jump, n_windows):
        """numpy.sum(arr[s:s + window_size]) for s = k * window_jump, k < n_windows, on the device (mg_window_sums)."""
        import ctypes
        if arr.dtype.kind not in "bui":
            raise NotImplementedError("the device path sums boolean and integer position_dics only (dtype %s)" % arr.dtype)
        if arr.dtype.itemsize == 1 and arr.dtype.kind in "bu":
            vals, elem = np.ascontiguousarray(arr).view(np.uint8), 1
        else:
            vals, elem = np.ascontiguousarray(arr, dtype=np.int64), 8
        sums = np.empty(n_windows, dtype=np.int64)
        _lib.require_device(_device())
        _lib.check(_lib.lib.mg_window_sums(_device(), ctypes.c_void_p(vals.ctypes.data) if vals.size else None, elem, vals.size,
                                           window_size, window_jump, n_windows, ctypes.c_void_p(sums.ctypes.data), None))
        return sums.astype(np.uint64) if arr.dtype.kind == "u" else sums       # numpy.sum's result type

    def sliding_window_calculate(self, window_size, window_jump=1, operation="sum", output="dict", threshold=1,
                                 seqs_to_exclude=[]):
        """genome.py:1036-1100.  operation may be "sum", "average", or "set". Output may be "dict", "coords",
        "annotation_set" or a file-like object.  Quirks kept: the last `window_size` positions never start a window, a new
        region is compared by WINDOW INDEX against the previous region's end COORDINATE, "coords" cannot work (the
        reference misspells `threshold`)."""
        is_file = hasattr(output, "write")
        if output == "dict":
            new_dic = {}
        elif output == "annotation_set":
            annotation_set = AnnotationSet()
            annotation_set.region = {}
        elif output == "coords":
            coords_list = []
        for seqid in self:
            arr = self[seqid]
            if len(arr) > window_size and seqid not in seqs_to_exclude:
                if output == "dict":
                    new_dic[seqid] = []
                coords_list = []
                n_windows = len(range(len(arr))[:-1 * window_size]) // window_jump
                if operation == "set":
                    for position in range(n_windows):
                        window_start = position * window_jump
                        new_dic[seqid].append(set(arr[window_start:window_start + window_size].tolist()))
                else:
                    sums = self._window_sums(arr, window_size, window_jump, n_windows) if n_windows > 0 else np.zeros(0, np.int64)
                    if operation == "sum":
                        values = sums
                    elif operation == "average":
                        values = sums * 1.0 / window_size
                    if n_windows > 0 and operation not in ("sum", "average"):
                        raise UnboundLocalError("local variable 'value' referenced before assignment")
                    if output == "dict":
                        new_dic[seqid].extend(list(values))
                    elif output == "annotation_set":
                        above = np.asarray(values >= threshold)
                        edges = np.flatnonzero(np.diff(np.concatenate(([False], above, [False])).astype(np.int8)))
                        for first, past in zip(edges[0::2].tolist(), edges[1::2].tolist()):
                            # window `first` is the first of a run at or above the threshold, `past` the first below again
                            if len(coords_list) == 0 or first > coords_list[-1][1]:
                                coords_list.append([1 + first * window_jump])
                            if past < n_windows:
                                if len(coords_list[-1]) == 1:
                                    coords_list[-1].append(past * window_jump + window_size)
                                else:
                                    coords_list[-1][1] = past * window_jump + window_size
                    elif output == "coords":
                        if n_windows > 0:
                            if bool(np.any(threshold[0] <= values)):
                                raise NameError("global name 'thredshold' is not defined")
                    elif is_file:
                        output.write("".join(seqid + '\t' + _py2_str(v.item()) + '\n' for v in values))
                    if verbose:
                        step = 10000000 // np.gcd(10000000, window_jump)
                        for position in range(0, n_windows, int(step)):
                            print("processed " + seqid + " to position " + str(position))
                if output == "annotation_set":
                    if len(coords_list) > 0:
                        if len(coords_list[-1]) == 1:
                            coords_list[-1].append(len(arr))
                        for coords in coords_list:
                            ID = seqid + "-window" + str(coords[0])
                            annotation_set.region[ID] = BaseAnnotation(ID, seqid, tuple(coords), "region", annotation_set=annotation_set)
                if verbose:
                    print("processed " + seqid)
                    if output == 'annotation_set':
                        for region in _order(list(annotation_set.region)):
                            if annotation_set.region[region].seqid == seqid:
                                print(str(annotation_set.region[region].coords))
        if output == "dict":
            return {k: new_dic[k] for k in _order(list(new_dic))}        # a Python-2.7 dict filled in this order
        elif output == "annotation_set":
            # the reference returns copy.deepcopy(annotation_set): the region table ends up re-inserted in slot order
            annotation_set.region = {k: annotation_set.region[k] for k in _order(list(annotation_set.region), deepcopy=True)}
            _DEEPCOPIED_SETS.add(annotation_set)
            return annotation_set
        elif output == "coords":
            return coords_list


# ---------------------------------------------------------------------------------------------
# Genome (genome.py:880-978)
# ---------------------------------------------------------------------------------------------

class Genome(object):
    """genome class: sequence + annotations (genome.py:880)."""

    def __init__(self, genome_sequence=None, annotations=None, varients=None, annotation_format='annotation_set',
                 truncate_names=False):
        if genome_sequence.__class__.__name__ == 'GenomeSequence' or genome_sequence is None:
            self.genome_sequence = genome_sequence
        else:
            self.genome_sequence = GenomeSequence(genome_sequence, truncate_names=truncate_names)
        if annotations is not None:
            # genome.py:889 tests for the misspelt class name "AnotationSet", so an AnnotationSet object is
            # never attached by the reference constructor; mirrored (the attribute is simply not set).
            if annotations.__class__.__name__ == "AnotationSet" and annotation_format == 'annotation_set':
                self.annotations = annotations
                self.annotations.genome = self
            elif annotation_format == 'gff3':
                self.annotations = read_gff(annotations)
                self.annotations.genome = self
            elif annotation_format == 'blast_csv':
                self.annotations = read_blast_csv(annotations)
                self.annotations.genome = self
            elif annotation_format == 'exonerate_output':
                self.annotations = read_exonerate(annotations)
                self.annotations.genome = self
            elif annotation_format == 'cegma_gff':
                self.annotations = read_cegma_gff(annotations)
                self.annotations.genome = self
        else:
            self.annotations = annotations

    def get_scaffold_fasta(self, seqid):
        return '>' + seqid + '\n' + self.genome_sequence[seqid]

    def get_genome_fasta(self, remove_spaces=False):
        fasta_list = []
        for seqid in self.genome_sequence:
            fasta_header = seqid.split()[0] if remove_spaces else seqid
            fasta_list.append('>' + fasta_header + '\n' + self.genome_sequence[seqid])
        return "\n".join(fasta_list)

    def get_seqids(self, from_annotations=False):
        seqid_list = []
        warning = False
        if self.genome_sequence is not None:
            for seqid in self.genome_sequence:
                seqid_list.append(seqid)
        if self.annotations is not None and from_annotations:
            for seqid in self.annotations.get_all_seqids():
                if seqid not in seqid_list:
                    seqid_list.append(seqid)
                    warning = True
        if warning:
            print("warning, some annotations possessed seqids not found in sequence dictionary")
        return seqid_list

    def read_gff(self, gff, *args, **kwargs):
        if getattr(self, "annotations", None) is not None:
            self.annotations.read_gff(gff, *args, **kwargs)
        else:
            self.annotations = read_gff(gff, *args, **kwargs)
            self.annotations.genome = self

    def read_exonerate(self, exonerate_output):
        """genome.py:950-955"""
        if getattr(self, "annotations", None) is not None:
            self.annotations.read_exonerate(exonerate_output)
        else:
            self.annotations = read_exonerate(exonerate_output)
            self.annotations.genome = self

    def read_cegma_gff(self, cegma_gff):
        """genome.py:963-968"""
        if getattr(self, "annotations", None) is not None:
            self.annotations.read_cegma_gff(cegma_gff)
        else:
            self.annotations = read_cegma_gff(cegma_gff)
            self.annotations.genome = self

    def read_blast_csv(self, blast_csv, hierarchy=['match', 'match_part'], source='blast', find_truncated_locname=False):
        """genome.py:957-961"""
        if getattr(self, "annotations", None) is None:
            self.annotations = AnnotationSet()
            self.annotations.genome = self
        self.annotations.read_blast_csv(blast_csv, hierarchy=hierarchy, source=source, find_truncated_locname=find_truncated_locname)
