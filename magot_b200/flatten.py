"""Host-side flattener: annotation objects -> SoA interval tables in reference emission order.

This is the host half of ParentAnnotation.get_fasta (genome.py:677-731) and
AnnotationSet.get_fasta (genome.py:578-582): it reproduces WHICH intervals are emitted, in WHICH
order, under WHICH header -- per transcript the children are keyed by their coords (identical
coords collapse, last one wins), sorted ascending by (start, end) and reversed when the LAST
child's strand is '-'; each child is reverse-complemented by its OWN strand -- and leaves every
byte of sequence work (slicing with Python clamp semantics, reverse complement, join, translation,
FASTA framing) to the device.
"""
import numpy as np

from . import engine


class _Top(object):
    __slots__ = ("entries", "longest", "genomic")

    def __init__(self, entries, longest, genomic):
        self.entries = entries          # list of entries; an entry is a list of leaf-record ids
        self.longest = longest
        self.genomic = genomic


def _short_circuits(obj):
    """ParentAnnotation.get_fasta returns "" before it looks at `longest` (genome.py:683, :730-731): no children, no set, no genome."""
    return not (len(obj.child_list) > 0 and obj.annotation_set is not None) or obj.annotation_set.genome is None


class Flattener(object):
    def __init__(self, annotation_set):
        self.aset = annotation_set
        self.gs = annotation_set.genome.genome_sequence
        self.index = annotation_set.build_index()       # cached on the set between calls (see AnnotationSet.build_index)
        self.tops = []
        # leaf records
        self.names = []                 # header text without '>' (str)
        self.rec_seg_off = [0]
        self.rec_phase = []
        self.seg_contig = []
        self.seg_start = []
        self.seg_end = []
        self.seg_strand = []
        self._contig_cache = {}

    # -- collection ------------------------------------------------------------------------------
    def _contig(self, seqid):
        c = self._contig_cache.get(seqid)
        if c is None:
            try:
                c = self.gs.contig_index(seqid)
            except Exception:
                # BaseAnnotation.get_seq prints and returns None (genome.py:611-614); the caller's
                # "".join then raises TypeError (genome.py:705)
                print("either base_annotation has not annotation_set, or annotation_set has no genome, or genome has no"
                      "            genome sequence, or genome sequence has no matching seqid, or coords are out of range on that seqid")
                print(seqid)
                raise TypeError("sequence item 0: expected string, NoneType found")
            self._contig_cache[seqid] = c
        return c

    def _leaf(self, name, segs, phase=0):
        rid = len(self.names)
        self.names.append(name)
        for (contig, start, end, minus) in segs:
            self.seg_contig.append(contig)
            self.seg_start.append(start)
            self.seg_end.append(end)
            self.seg_strand.append(minus)
        self.rec_seg_off.append(len(self.seg_contig))
        self.rec_phase.append(phase)
        return rid

    def _collect(self, obj, name_from):
        """Entries of obj.get_fasta(...) before the `longest` selection (genome.py:683-719)."""
        from .genome import BaseAnnotation
        if not (len(obj.child_list) > 0 and obj.annotation_set is not None):
            return []
        if obj.annotation_set.genome is None:
            return []
        index = self.index
        first = index[obj.child_list[0]]
        if isinstance(first, BaseAnnotation):
            child_dict = {}
            strand = None
            for child in obj.child_list:
                co = index[child]
                if isinstance(co, BaseAnnotation):
                    child_dict[co.coords] = co
                else:
                    print("ParentAnnotation has both ParentAnnotation and BaseAnnotation children!")
                    print(obj.ID)
                strand = co.strand
            order = sorted(child_dict)
            if strand == '-':
                order.reverse()
            segs = []
            phase = 0
            for k, c in enumerate(order):
                co = child_dict[c]
                if co.strand == '+' or co.strand == '.':
                    minus = 0
                elif co.strand == '-':
                    minus = 1
                else:
                    print(co.ID + ' has invalid strand value "' + co.strand + '"')
                    raise TypeError("sequence item %d: expected string, NoneType found" % k)
                segs.append((self._contig(co.seqid), c[0], c[1], minus))
                if k == 0:
                    phase = getattr(co, "phase", 0) or 0
            return [[self._leaf(obj.__dict__[name_from], segs, phase)]]
        entries = []
        for child in obj.child_list:
            co = index[child]
            if isinstance(co, BaseAnnotation):
                print("ParentAnnotation has both ParentAnnotation and BaseAnnotation children!")
                print(obj.ID)
                continue
            sub = self._collect(co, name_from)
            leaves = [rid for entry in sub for rid in entry]
            if leaves:
                entries.append(leaves)
        return entries

    def add_top(self, obj, seq_type="nucleotide", longest=False, genomic=False, name_from='ID'):
        if genomic is True:                                           # genome.py:680-682
            c = obj.get_coords()                                      # None -> TypeError below, as the reference
            rid = self._leaf(obj.ID, [(self._contig(obj.seqid), c[0], c[1], 0)])
            self.tops.append(_Top([[rid]], False, True))
            return
        # a top that short-circuits never reaches the `longest` selection (its max() over no sequences would raise ValueError)
        self.tops.append(_Top(self._collect(obj, name_from), longest is True and not _short_circuits(obj), False))

    # -- execution -------------------------------------------------------------------------------
    def _table(self, rec_ids, pre, suf):
        """RecordTable over the chosen leaf records (rec_ids may contain -1 = record without segments)."""
        seg_off = np.asarray(self.rec_seg_off, dtype=np.int64)
        ids = np.asarray(rec_ids, dtype=np.int64)
        valid = ids >= 0
        safe = np.minimum(np.maximum(ids, 0), seg_off.size - 2) if seg_off.size > 1 else np.zeros_like(ids)
        lo = np.where(valid, seg_off[safe], 0)
        hi = np.where(valid, seg_off[np.minimum(safe + 1, seg_off.size - 1)], 0)
        cnt = hi - lo
        rec_seg_off = np.concatenate(([0], np.cumsum(cnt)))
        total = int(rec_seg_off[-1])
        # gather segment rows: positions lo[r] .. hi[r]-1 for every record
        rep = np.repeat(np.arange(ids.size), cnt)
        within = np.arange(total) - np.repeat(rec_seg_off[:-1], cnt)
        src = lo[rep] + within
        sc = np.asarray(self.seg_contig, dtype=np.int32)
        ss = np.asarray(self.seg_start, dtype=np.int64)
        se = np.asarray(self.seg_end, dtype=np.int64)
        st = np.asarray(self.seg_strand, dtype=np.int8)
        ph = np.asarray(self.rec_phase, dtype=np.int8)
        # literals: prefix bytes immediately followed by suffix bytes, record after record (no Python statement per record)
        n = ids.size
        pre_len = np.fromiter(map(len, pre), dtype=np.int32, count=n)
        suf_len = np.fromiter(map(len, suf), dtype=np.int32, count=n)
        both = pre_len.astype(np.int64) + suf_len
        lit_off = np.concatenate(([0], np.cumsum(both)[:-1])) if n else np.zeros(0, dtype=np.int64)
        blob = b"".join(x for pair in zip(pre, suf) for x in pair)
        lit = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(0, dtype=np.uint8)
        return engine.RecordTable(rec_seg_off, sc[src] if total else sc[:0], ss[src] if total else ss[:0],
                                  se[src] if total else se[:0], st[src] if total else st[:0], lit_off, pre_len,
                                  suf_len, lit, np.where(valid, ph[safe] if ph.size else 0, 0).astype(np.int8))

    def run(self, seq_type, codon64=None):
        tbl, rec_ids, protein = self.records(seq_type)
        if tbl is None:
            return ""
        eng = self.gs._engine()
        text, l2 = eng.run_table(tbl, protein=protein, want_lengths=protein, codon64=codon64)
        if protein and l2 is not None and (l2[1] < 0)[np.asarray(rec_ids) >= 0].any():
            # Sequence.translate returned None (spliced length <= 2): '>' + name + '\n' + None (genome.py:710)
            raise TypeError("cannot concatenate 'str' and 'NoneType' objects")
        return engine.decode_text(text, strip_last=1)

    def records(self, seq_type):
        """(RecordTable, leaf id per record (-1 = blank line), protein) of what run(seq_type) prints, or (None, [], False)
        without tops.  The `longest` selection runs here (one length pass on the device)."""
        if seq_type not in ("nucleotide", "protein"):
            if any(t.entries for t in self.tops if not t.genomic):
                print(seq_type + ' is not valid seq_type. Please specify "protein" or "nucleotide".')
                raise UnboundLocalError("local variable 'new_seq' referenced before assignment")
        if not self.tops:
            return None, [], False
        eng = self.gs._engine()
        any_longest = any(t.longest for t in self.tops)
        # genomic records are always nucleotide text (genome.py:680-682 ignores seq_type); they cannot be
        # mixed with protein records in one call (AnnotationSet.get_fasta passes one flag to every object)
        protein = (seq_type == "protein") and not all(t.genomic for t in self.tops)
        lens = None
        if any_longest:
            n = len(self.names)
            if n:
                tbl = self._table(list(range(n)), [b""] * n, [b""] * n)
                _, (nuc_len, aa_len) = eng.run_table(tbl, protein=protein, want_lengths=True)
                lens = aa_len if protein else nuc_len
        rec_ids, pre, suf = [], [], []
        for top in self.tops:
            entries = top.entries
            if top.longest:
                seqlens = {}
                for e in entries:                                   # genome.py:720-724, last among equals wins
                    L = 0
                    for k, rid in enumerate(e):
                        if lens[rid] < 0:
                            raise TypeError("cannot concatenate 'str' and 'NoneType' objects")
                        L += int(lens[rid]) + (0 if k == 0 else 1 + len(self.names[rid]))
                    seqlens[L] = e
                if not seqlens:
                    raise ValueError("max() arg is an empty sequence")
                entries = [seqlens[max(seqlens)]]
            leaves = [rid for e in entries for rid in e]
            if not leaves:
                rec_ids.append(-1)                                   # "" in the joined list -> blank line
                pre.append(b"")
                suf.append(b"\n")
                continue
            for rid in leaves:
                rec_ids.append(rid)
                pre.append(b">" + self.names[rid].encode("latin-1") + b"\n")
                suf.append(b"\n\n" if top.genomic else b"\n")
        return self._table(rec_ids, pre, suf), rec_ids, protein
