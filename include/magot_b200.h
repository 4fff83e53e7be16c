/* magot_b200.h -- C ABI of libmagot_b200.so: the B200 (sm_100a) implementation of MAGOT's
 * annotation-driven sequence path (FASTA + GFF3/GTF -> spliced CDS/transcript nucleotides ->
 * reverse complement -> protein -> six-frame/ORF scan).
 *
 * The reference (pure Python 2.7, /root/reference/genome.py) has no FFI layer; its boundary is
 * the Python API.  Every entry point below therefore cites the reference function(s) whose work
 * it replaces; `magot_b200/genome.py` binds them with ctypes behind the unchanged Python API and
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a negative
 * MG_E* code, with a thread-local message available from mg_last_error(); no exceptions, no
 * callbacks.  The caller owns every buffer it passes; the library owns what sits behind a handle.
 * `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream).  A handle is
 * bound to one CUDA device; calls on one handle must be serialised by the caller, different
 * handles/devices may be driven from different host threads.  There is NO CPU fallback: without
 * a CUDA device every compute entry point fails with MG_ECUDA.
 */
#ifndef MAGOT_B200_H
#define MAGOT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MG_VERSION 100            /* 0.1.0 */

enum {
    MG_OK = 0,
    MG_EINVAL = -1,               /* bad argument */
    MG_ECUDA = -2,                /* CUDA runtime error / no device */
    MG_ENOMEM = -3,
    MG_ESTATE = -4                /* call order violated (e.g. emit before prepare) */
};

typedef struct mg_genome mg_genome;   /* device-resident packed genome            */
typedef struct mg_plan mg_plan;       /* device-resident interval/record tables   */

/* ---- introspection ---------------------------------------------------------------------- */
int mg_version(void);
const char *mg_last_error(void);
int mg_device_count(int *n_out);

/* ---- K0: genome storage -- replaces GenomeSequence.__init__ (genome.py:856-877, storage only)
 * The genome lives on the device as one nibble per base (0.5 B/base):
 *   0-3 = A C G T, 4-7 = a c g t, 8 = N, 9 = n, 10 = '-', 11-14 = R Y K M, 15 = "exception":
 * any other byte (the reference keeps every FASTA byte verbatim on '+' strand output,
 * genome.py:606) is recorded in a sorted (position, byte) side list.                         */
int mg_genome_create(int device, int64_t n_contigs, const int64_t *contig_len, mg_genome **out);
/* Pack `n` ASCII bytes (newlines already removed) of contig `contig` starting at 0-based
 * `offset` inside it.  `ascii` is a HOST pointer (pinned or pageable); `offset` must be a
 * multiple of 32 unless it ends the contig.  Chunks may arrive in any order.                */
int mg_genome_pack(mg_genome *g, int64_t contig, int64_t offset, const uint8_t *ascii, int64_t n, void *stream);
/* Same, from a DEVICE pointer (used when the text is produced on the device).               */
int mg_genome_pack_device(mg_genome *g, int64_t contig, int64_t offset, const uint8_t *ascii_dev, int64_t n, void *stream);
/* K0f: the same from the RAW body of a FASTA record (`raw` = host bytes between the header line and the next
 * header, line ends included): CR and LF are dropped on the device by a single-pass stream compaction, every other
 * byte is kept -- replaces `seq = seq + line.replace('\n','').replace('\r','')` (genome.py:875) so that the host
 * never touches the sequence bytes.  The number of kept bytes must equal the contig length given to
 * mg_genome_create (count the line ends on the host), else MG_EINVAL.                          */
int mg_genome_pack_fasta(mg_genome *g, int64_t contig, const uint8_t *raw, int64_t n_raw, void *stream);
/* Host helper of the FASTA header scan: out[r] = number of CR / LF bytes in data[lo[r], hi[r]) for every record body, so that
 * the contig lengths (body bytes minus line ends, genome.py:875) are known before mg_genome_create without a Python pass over
 * the sequence bytes.  Threaded; no GPU work.                                                                             */
int mg_count_line_ends(const uint8_t *data, int64_t n, int64_t n_ranges, const int64_t *lo, const int64_t *hi, int64_t *out);
/* Sort the exception list and make the genome usable by every call below.
 * Every call that can change the bases -- mg_genome_pack*, mg_genome_finalize, mg_genome_mask -- makes the results of an
 * earlier count (mg_sixframe_count*, mg_orfcall_count) or plan prepare (mg_plan_prepare*) stale: their emits then fail with
 * MG_ESTATE until the count or prepare is repeated.  A CUDA graph replays what it captured without these host checks, so a
 * graph captured before such a call must not be replayed after it.                                                        */
int mg_genome_finalize(mg_genome *g, int64_t *n_exceptions_out);
int mg_genome_destroy(mg_genome *g);
int64_t mg_genome_bytes(const mg_genome *g);          /* device bytes held by the handle      */
/* Decode contig[lo:hi) (0-based, half open, already clamped) back to the exact FASTA bytes;
 * minus != 0 gives Sequence.reverse_compliment of it (genome.py:784-793).  Backs
 * GenomeSequence.__getitem__/slicing, coords2fasta (genome_tools.py:656-661),
 * get_scaffold_fasta (genome.py:907) and BaseAnnotation.get_seq (genome.py:603-608).        */
int mg_genome_fetch(mg_genome *g, int64_t contig, int64_t lo, int64_t hi, int minus, uint8_t *out_host, void *stream);

/* ---- K5: interval scatter -- replaces the list surgery of mask_from_gff (genome_tools.py:394-428).
 * Intervals are 0-based half-open [lo, hi) on `contig`, already clamped like the Python slice
 * [start-1:stop]; they may overlap.  hard = 0: lower-case them (soft mask); hard = 1: replace them
 * by 'N'.  upper_first != 0 upper-cases the whole genome before (overwrite_softmask, :403-404).
 * Both planes and the exception list are updated; the handle stays finalized.  Counts and prepared plans of this genome
 * become stale (see mg_genome_finalize).  On an argument error (MG_EINVAL) the genome is left unchanged.                */
int mg_genome_mask(mg_genome *g, int64_t n_intervals, const int32_t *contig, const int64_t *lo, const int64_t *hi,
                   int hard, int upper_first, void *stream);

/* ---- K6: per-base flags and sliding-window sums -- the device side of position_dic (genome.py:981-1100).
 * mg_genome_at_flags: out_host[i] = 1 where base lo+i of `contig` is one of "ATat", else 0
 *   (position_dic.at_content, genome.py:1030-1034); lo must be a multiple of 8.
 * mg_window_sums: sums_host[k] = sum(values[k*jump : k*jump + window]) for k < n_windows, slices clamped at n like
 *   numpy's (numpy.sum at genome.py:1055) -- one single-pass prefix scan (warp/block scans + decoupled look-back) and
 *   one gather per window instead of n_windows * window additions.  elem_size 1 = uint8 / numpy bool, 8 = int64.  */
int mg_genome_at_flags(mg_genome *g, int64_t contig, int64_t lo, int64_t hi, uint8_t *out_host, void *stream);
int mg_window_sums(int device, const void *values_host, int elem_size, int64_t n, int64_t window, int64_t jump,
                   int64_t n_windows, int64_t *sums_host, void *stream);

/* ---- K1: interval tables -- replaces the per-child work of ParentAnnotation.get_fasta
 * (genome.py:687-705) and the slice arithmetic of BaseAnnotation.get_seq (genome.py:603-608).
 * A plan is a list of n_rec output records.  Record r owns segments
 * [rec_seg_off[r], rec_seg_off[r+1]) ALREADY in the reference's emission order (sorted by
 * coords, duplicates collapsed, reversed when the last child's strand is '-'), plus a literal
 * prefix (e.g. ">ID\n") and suffix (e.g. "\n") taken from `lit` at rec_lit_off[r]
 * (prefix bytes immediately followed by suffix bytes).
 * Segment coordinates are the raw, sorted GFF pair (start,end), 1-based inclusive; the device
 * applies Python slice semantics contig[start-1:end] including negative / out-of-range values.
 * A segment may be of any length (a whole chromosome of more than 2^31 bases too).  A record's
 * payload (its clamped segments together) is limited to 3 * (2^31 - 1) + 2 bases, so that its
 * protein has at most 2^31 - 1 residues: a longer record fails with MG_EINVAL.
 * seg_strand: 0 = '+' or '.', 1 = '-' (reverse-complement that segment).
 * rec_phase (may be NULL): phase of the first segment in emission order, used only with
 * MG_PROT_USE_PHASE.                                                                          */
int mg_plan_create(mg_genome *g, int64_t n_rec, const int64_t *rec_seg_off,
                   int64_t n_seg, const int32_t *seg_contig, const int64_t *seg_start,
                   const int64_t *seg_end, const int8_t *seg_strand,
                   const int64_t *rec_lit_off, const int32_t *rec_pre_len, const int32_t *rec_suf_len,
                   const uint8_t *lit, int64_t n_lit, const int8_t *rec_phase,
                   void *stream, mg_plan **out);
int mg_plan_destroy(mg_plan *p);

/* flags for mg_plan_prepare / emit */
#define MG_PROT_TRIMX      1      /* Sequence.translate(trimX=True): drop ONE leading 'X' (genome.py:819-821) */
#define MG_PROT_USE_PHASE  2      /* non-reference extension: start at the GFF phase of the first segment     */
#define MG_PROT_DEFER      4      /* mg_plan_prepare_async only: leave out the record pass (amino-acid counts, protein offsets);
                                     mg_plan_prepare_prot_async runs it later -- on another stream next to K2, or never when only
                                     the nucleotide text is wanted (e.g. the exon-based transcripts of gff2fasta)          */

/* Clamp, measure and scan (warp/block prefix sums on the device).  Outputs (host, may be NULL):
 * total bytes of the nucleotide text and of the protein text (literals included).
 * Must be called once before any emit; everything stays on the device.  The record pass reads the genome (trimX of the first
 * codon) and the emits read it again, so a prepare holds for the genome as it was: after a pack, finalize or mask of the
 * plan's genome, mg_plan_prepare_prot_async, mg_plan_totals, mg_plan_lengths and every mg_emit_* of the plan fail with
 * MG_ESTATE until it is prepared again.                                                                              */
int mg_plan_prepare(mg_plan *p, int prot_flags, int64_t *nuc_total, int64_t *prot_total, void *stream);
/* The same without the host round trip, for callers that already hold buffers: nuc_capacity / prot_capacity are the sizes
 * the caller's nucleotide / protein output buffers can take (an upper bound is sum(max(0, end-start+1)) + framing bytes,
 * resp. a third of it + framing).  K1, K2 and K3 can then be queued back to back on the stream (or captured in a CUDA
 * graph): the tile counts are derived on the device and surplus CTAs exit.  mg_plan_totals waits for the stream and
 * returns the real sizes; it fails if they exceeded the capacities (the texts are then truncated).             */
int mg_plan_prepare_async(mg_plan *p, int prot_flags, int64_t nuc_capacity, int64_t prot_capacity, void *stream);
int mg_plan_prepare_prot_async(mg_plan *p, void *stream);   /* the record pass left out by MG_PROT_DEFER; after the piece pass in stream order */
int mg_plan_totals(mg_plan *p, int64_t *nuc_total, int64_t *prot_total, void *stream);
/* Per-record payload lengths to the host (for `longest=True`, genome.py:720-724).
 * nuc_len[r] = spliced bases; aa_len[r] = amino acids, or -1 where the reference's translate
 * returns None (spliced length <= 2, genome.py:810).  Either pointer may be NULL.           */
int mg_plan_lengths(mg_plan *p, int64_t *nuc_len, int64_t *aa_len, void *stream);
/* Genetic code of the plan's protein text (K3, K23, mg_emit_products_*, every _host variant): codon64[16*b0 + 4*b1 + b2]
 * (A=0 C=1 G=2 T=3) is the residue of codon b0 b1 b2, '*' a stop; no entry may be 'X' (a codon with a base outside ACGT is 'X'
 * whatever the code, which is what trimX tests).  The table is uploaded by this call, so emits captured in a CUDA graph
 * afterwards stay valid.  codon64 == NULL restores the genome's standard code (NCBI table 1).                                 */
int mg_plan_set_codon_table(mg_plan *p, const uint8_t *codon64);

/* ---- K2: spliced nucleotides (+ per-segment reverse complement, + literal framing) ---------
 * replaces ParentAnnotation.get_fasta seq_type="nucleotide" (genome.py:687-710) and
 * Sequence.reverse_compliment (genome.py:784-793).  `out_dev` must be 32-byte aligned and hold
 * nuc_total rounded up to a multiple of 32 bytes (each lane issues one 256-bit store).                                            */
int mg_emit_nuc_device(mg_plan *p, uint8_t *out_dev, void *stream);
/* ---- K3: protein -- replaces Sequence.translate(frame=0,strand='+') (genome.py:795-822) on the
 * spliced sequence (genome.py:707).  Same buffer rules with prot_total.                     */
int mg_emit_prot_device(mg_plan *p, uint8_t *out_dev, void *stream);
/* ---- K23: fused splice + translate -- the reference translates the very string it has just joined (genome.py:704-707:
 * seq = "".join(...get_seq()); Sequence(seq).translate()).  One launch writes the nucleotide text of the plan to nuc_out_dev and
 * its protein text to prot_out_dev (buffer rules of the two single calls): the CTA that assembles 32 KB of nucleotide text keeps
 * the bases in shared memory and translates the codons that start there, so the genome is read once.  Bit-identical to
 * mg_emit_nuc_device + mg_emit_prot_device.  The _host variant copies both texts to host buffers (stream-ordered).          */
int mg_emit_nuc_prot_device(mg_plan *p, uint8_t *nuc_out_dev, uint8_t *prot_out_dev, void *stream);
int mg_emit_nuc_prot_host(mg_plan *p, uint8_t *nuc_out_host, uint8_t *prot_out_host, void *stream);
/* ---- K2 + K2 + K3 of one batch in ONE launch -- what `gff2fasta` run three times (seq_type nucleotide on the exon-based
 * transcripts, nucleotide and protein on the CDS; genome_tools.py:324-330, genome.py:687-710) reads from the genome: the same
 * bases.  Nucleotide text of plan `pa` -> out_a, nucleotide text of plan `pb` -> out_b_nuc, protein text of `pb` -> out_b_prot
 * (buffer rules as above; any output may be NULL and is then skipped).  The tiles of the products are interleaved so that every
 * product advances through the record list at the same pace, `pb` slightly behind `pa`: when both plans list the same
 * transcripts in the same order (exon table / CDS table) the later products find their genome bytes in L2 instead of DRAM.
 * The texts are bit-identical to the single-product calls.                                                                */
int mg_emit_products_device(mg_plan *pa, uint8_t *out_a, mg_plan *pb, uint8_t *out_b_nuc, uint8_t *out_b_prot, void *stream);
int mg_emit_products_host(mg_plan *pa, uint8_t *out_a_host, mg_plan *pb, uint8_t *out_b_nuc_host, uint8_t *out_b_prot_host, void *stream);
/* Host-buffer variants: run the kernel into a library-owned device buffer and copy the exact
 * text (nuc_total / prot_total bytes) to `out_host` (pinned for full PCIe speed).  The copy is
 * stream-ordered; call mg_stream_sync before reading.                                        */
int mg_emit_nuc_host(mg_plan *p, uint8_t *out_host, void *stream);
int mg_emit_prot_host(mg_plan *p, uint8_t *out_host, void *stream);

/* ---- Sequence ops on arbitrary strings -----------------------------------------------------
 * mg_revcomp: Sequence.reverse_compliment (genome.py:784-793) of n host bytes.
 * mg_translate_ascii: Sequence.translate(frame, strand, trimX) (genome.py:795-822) of n_seq
 * strings stored back to back (seq i = in[off[i], off[i+1])), all with the same parameters --
 * backs cds2pep (genome_tools.py:664-675).  out_off[n_seq+1] receives the offsets of the results
 * in `out` (capacity out_cap bytes; (n+2)/3 + n_seq always suffices); out_len[i] = -1 where
 * the reference returns None.                                                                */
int mg_revcomp(int device, const uint8_t *in_host, int64_t n, uint8_t *out_host, void *stream);
int mg_translate_ascii(int device, const uint8_t *in_host, const int64_t *off, int64_t n_seq,
                       int frame, int minus, int trimX, uint8_t *out_host, int64_t out_cap,
                       int64_t *out_off, int64_t *out_len, void *stream);
/* Same with the caller's codon table: codon64[16*b0 + 4*b1 + b2] (A=0 C=1 G=2 T=3) is the byte emitted for the codon
 * b0 b1 b2 ('X' where the library has no entry) -- Sequence.translate(library=...) (genome.py:795, :814-817).
 * codon64 == NULL selects the reference's default table.                                      */
int mg_translate_ascii_table(int device, const uint8_t *codon64, const uint8_t *in_host, const int64_t *off, int64_t n_seq,
                             int frame, int minus, int trimX, uint8_t *out_host, int64_t out_cap, int64_t *out_off,
                             int64_t *out_len, void *stream);

/* ---- K4: six-frame translation + ORF scan -- replaces Sequence.get_orfs (genome.py:824-851)
 * over whole contigs [contig_lo, contig_hi).  Streams are visited in the reference's order
 * (frame 0 '-', 0 '+', 1 '-', 1 '+', 2 '-', 2 '+'; genome.py:829-830) with its frame quirk;
 * each translation is split on '*'; ORFs shorter than min_aa are dropped (0 == reference,
 * empty strings included).  Pass 1 counts, pass 2 emits.                                    */
typedef struct {
    int32_t contig;
    int8_t frame;                 /* 0,1,2 : the `frame` argument of translate()              */
    int8_t minus;                 /* 1 = translated from the reverse complement               */
    int16_t pad;
    int64_t start;                /* index of the ORF's first residue in that translation     */
    int64_t len;                  /* residues                                                 */
    int64_t aa_off;               /* offset of its text in the emitted amino-acid buffer      */
} mg_orf;
int mg_sixframe_count(mg_genome *g, int64_t contig_lo, int64_t contig_hi, int64_t min_aa,
                      int64_t *n_orf, int64_t *n_bytes, void *stream);
/* The same for a LIST of contigs in any order (e.g. one GPU's share of a length-balanced split): ORFs are emitted contig by
 * contig in list order.                                                                        */
int mg_sixframe_count_list(mg_genome *g, int64_t n_list, const int64_t *contig_ids, int64_t min_aa,
                           int64_t *n_orf, int64_t *n_bytes, void *stream);
/* The same two scans under another genetic code: codon64 as in mg_plan_set_codon_table.  A codon is a stop iff the table maps it
 * to '*' (any number of stop codons, 0..64); the following mg_sixframe_emit* writes residues from this table.  codon64 == NULL
 * is exactly mg_sixframe_count / mg_sixframe_count_list.  With the stop-codon index (mg_tune "six" = 2), a code whose stops
 * differ from TAA/TAG/TGA builds a second index (0.25 B/base, counted in mg_genome_bytes) next to the standard one; one such
 * index is kept, and pack / finalize / mask drop both.                                                                      */
int mg_sixframe_count_table(mg_genome *g, int64_t contig_lo, int64_t contig_hi, int64_t min_aa, const uint8_t *codon64,
                            int64_t *n_orf, int64_t *n_bytes, void *stream);
int mg_sixframe_count_list_table(mg_genome *g, int64_t n_list, const int64_t *contig_ids, int64_t min_aa, const uint8_t *codon64,
                                 int64_t *n_orf, int64_t *n_bytes, void *stream);
/* Emits the result of the preceding mg_sixframe_count on this genome handle.  aa_out_host gets
 * n_bytes residues (ORFs back to back, no separators), recs_host n_orf records.  Either may
 * be NULL.  *_device variant leaves the residues in `aa_out_dev` (16-byte aligned, n_bytes
 * rounded up to 16).  The residues are read from the genome at emit time: after a pack, finalize
 * or mask of the genome since the count, the emit fails with MG_ESTATE (count again).         */
int mg_sixframe_emit(mg_genome *g, uint8_t *aa_out_host, mg_orf *recs_host, void *stream);
int mg_sixframe_emit_device(mg_genome *g, uint8_t *aa_out_dev, mg_orf *recs_dev, void *stream);

/* ---- start-to-stop ORF calling (ORFfinder / getorf style) on whole contigs, both strands, three TRUE phases.
 * Phase p reads codons at offsets p, p+3, ... of the strand's 5'->3' sequence (the minus strand is the reverse complement,
 * phase counted from the contig's end); no frame quirk, no trimX.  Lower case is upper case; a codon with a base outside
 * A/C/G/T is neither a start nor a stop.  A stop is a codon that codon64 maps to '*'.  Each stop-bounded segment gives at most
 * one ORF: from its FIRST codon flagged in start64 through the stop that ends it (nested starts are not reported).  A segment
 * that runs to the contig end without a stop gives a 3' partial ORF, kept only when `partial` != 0.  The protein is the
 * translation of the start codon up to, not including, the stop, with the first residue always 'M'; ORFs of fewer than
 * min_aa residues are dropped.
 * Order: contig in list order, then stream in the order (phase 0 '-'), (0 '+'), (2 '-'), (2 '+'), (1 '-'), (1 '+') -- K4's
 * stream order, whose frames 1 and 2 read residue classes 2 and 1 -- then position (plus ascending, minus descending).
 * The count / emit state is the one mg_sixframe_count* uses: a count of either kind replaces the other, and an emit after the
 * other kind of count fails with MG_ESTATE.                                                                              */
typedef struct {
    int32_t contig;
    int8_t  minus;                /* 1 = minus strand                                                  */
    int8_t  phase;                /* 0..2, offset of the first codon in the strand's 5'->3' read       */
    int8_t  flags;                /* bit 0: no stop codon (3' partial)                                 */
    int8_t  start_codon;          /* 16*b0 + 4*b1 + b2, A=0 C=1 G=2 T=3                                */
    int64_t lo, hi;               /* 0-based half-open forward-contig interval, stop codon included    */
    int64_t len;                  /* residues, M included, stop excluded                               */
    int64_t aa_off;               /* offset of the residues in the emitted buffer                      */
} mg_orfcall;
/* codon64: as in mg_sixframe_count_table (NULL = table 1).  start64: 64 flags, byte 16*b0 + 4*b1 + b2 non-zero = start codon
 * (NULL = ATG only); at least one codon must be flagged and none may be a stop of codon64.  partial: report 3' partials.  */
int mg_orfcall_count(mg_genome *g, int64_t n_list, const int64_t *contig_ids, int64_t min_aa, const uint8_t *codon64,
                     const uint8_t *start64, int partial, int64_t *n_orf, int64_t *n_bytes, void *stream);
/* As mg_sixframe_emit / mg_sixframe_emit_device, for the preceding mg_orfcall_count (MG_ESTATE after a genome change too). */
int mg_orfcall_emit(mg_genome *g, uint8_t *aa_out_host, mg_orfcall *recs_host, void *stream);
int mg_orfcall_emit_device(mg_genome *g, uint8_t *aa_out_dev, mg_orfcall *recs_dev, void *stream);

/* ---- gene-model check of a prepared plan (start / stop codons, in-frame stops, reading frame, splice sites, codon usage).
 * Record r's payload S is its clamped segments in emission order, each reverse-complemented by its strand: the bytes the
 * nucleotide emit writes without framing.  skip = rec_phase[r] when MG_PROT_USE_PHASE is given and it is 0..2, else 0 (never
 * trimX).  Codon i is S[skip+3i, skip+3i+3) for i < n_codons = max(0, (len(S) - skip) / 3); rem = (len(S) - skip) mod 3, or 0
 * when len(S) <= skip.  A codon with a base outside A/C/G/T (either case) is ambiguous: never a start or a stop, not counted in
 * codon usage or GC.  A stop is a codon the plan's codon table (mg_plan_set_codon_table, default table 1) maps to '*'; a start is
 * a codon flagged in start64 (as in mg_orfcall_count).
 * Junction between segments k and k+1 of a record (caller's segment indices, emission order, both clamped like the plan and not
 * empty, same contig and strand): '+' intron [b_k, a_{k+1}), donor = bases b_k, b_k+1, acceptor = a_{k+1}-2, a_{k+1}-1; '-' intron
 * [b_{k+1}, a_k), donor = reverse complement of a_k-2, a_k-1, acceptor = reverse complement of b_{k+1}, b_{k+1}+1.  The intron
 * must hold at least 4 bases.  Class 1 = GT-AG, 2 = GC-AG, 3 = AT-AC, 4 = any other pair (case ignored, a base outside ACGT
 * gives 4), 0 = no junction (last segment, empty segment, contig or strand change, gap under 4 bases, overlap, wrong order).
 * The chunks mg_plan_create makes of a segment of 2^31 bases or more are not junctions.                                     */
typedef struct {
    int64_t nuc_len;              /* len(S)                                                                  */
    int64_t gc;                   /* G/C bases in unambiguous codons                                         */
    int32_t n_codons;
    int32_t n_ambig;              /* ambiguous codons                                                        */
    int32_t n_stop;               /* stop codons, the terminal one included                                  */
    int32_t first_stop;           /* codon index of the first stop, -1 = none                                */
    int32_t gc3;                  /* unambiguous codons whose third base is G or C                           */
    int32_t n_junction;           /* junctions of class 1..4                                                 */
    int32_t n_noncanonical;       /* junctions of class 4                                                    */
    int32_t flags;                /* MG_CHK_*                                                                */
    int8_t  skip;
    int8_t  rem;
    uint8_t start_codon;          /* 16*b0 + 4*b1 + b2 of codon 0, 0xFF = absent or ambiguous                 */
    uint8_t stop_codon;           /* the same for the last complete codon                                    */
    int32_t pad;
} mg_cds_check;                   /* 56 bytes                                                                */
#define MG_CHK_NO_START            1   /* codon 0 absent, ambiguous or not a start                                */
#define MG_CHK_NO_STOP             2   /* no complete codon, or the last one is not a stop                        */
#define MG_CHK_INTERNAL_STOP       4   /* a stop before the last codon (n_stop - terminal > 0)                     */
#define MG_CHK_PARTIAL_CODON       8   /* rem != 0                                                                 */
#define MG_CHK_NONCANONICAL_SPLICE 16  /* a junction of class 4                                                    */
#define MG_CHK_AMBIGUOUS           32  /* an ambiguous codon                                                       */
#define MG_CHK_EMPTY               64  /* n_codons == 0                                                            */
/* rec_out[n_rec]; codon_counts[64 * r + 16*b0 + 4*b1 + b2] (n_rec x 64, may be NULL: not computed); junction[e] = class of the
 * junction after caller segment e (n_seg entries of the table given to mg_plan_create, may be NULL).  flags: 0 or
 * MG_PROT_USE_PHASE.  start64 is a host table as in mg_orfcall_count (NULL = ATG), checked against the plan's code and passed to
 * the kernels by value.  Needs a plan prepared on the genome as it is (MG_ESTATE otherwise); MG_PROT_DEFER is enough.
 * mg_plan_check_device takes device pointers for the three outputs and queues everything on `stream` without a host round trip
 * (a CUDA graph can capture it); mg_plan_check takes host pointers and copies in stream order (sync before reading).
 * The stop set of the plan's code and the start set are passed to the kernels by value: a captured check keeps the genetic
 * code and the start codons it was captured with, whatever mg_plan_set_codon_table is called later (capture it again).                                                                                                              */
int mg_plan_check(mg_plan *p, int flags, const uint8_t *start64, mg_cds_check *rec_out, uint32_t *codon_counts, int8_t *junction,
                  void *stream);
int mg_plan_check_device(mg_plan *p, int flags, const uint8_t *start64, mg_cds_check *rec_out, uint32_t *codon_counts,
                         int8_t *junction, void *stream);

/* ---- CDS prediction of a prepared plan: the longest ORF of every record's spliced payload, mapped back to genome CDS segments
 * (TransDecoder.LongOrfs style, one ORF per record).  Record r's payload S is the one of mg_plan_check; n = len(S).
 * A codon starts at every position i with i + 3 <= n; its frame is i mod 3.  Case is ignored and a codon with a base outside
 * A/C/G/T is neither a start nor a stop.  A stop is a codon the plan's code (mg_plan_set_codon_table) maps to '*'; a start is a
 * codon flagged in start64 (NULL = ATG; at least one codon, no stop, as mg_orfcall_count checks it).
 * Stretches: in frame f the stops cut the codons f, f+3, ... into stretches.  A stretch ends at a stop (included) or at the
 * frame's last complete codon (an open 3' end); the first stretch of a frame begins at codon f (an open 5' end), every later
 * one right after a stop.  A stretch's ORF starts at its first start codon b -- with MG_PRED_5PARTIAL the first stretch of a
 * frame starts at its first codon instead, start codon or not -- and ends after the stop, or after the frame's last complete
 * codon for an open 3' end, which is kept only with MG_PRED_3PARTIAL.  n_aa counts the codons from the start up to, not
 * including, the stop; a candidate needs n_aa >= max(1, min_aa).  Type bit 0 (5' partial): the first codon is not a start
 * codon; bit 1 (3' partial): there is no stop.  Each record gets the candidate with the largest n_aa, ties broken by the
 * smallest start; a record without a candidate reports none (lo = hi = -1, n_aa = 0, frame = -1, type = 0, codons 0xFF).
 * Mapping: caller segment e of the record (the table given to mg_plan_create; the chunks it makes of a segment of 2^31 bases
 * or more are never visible), clamped as the plan clamps it to [cl, ch), covers payload range [o_e, o_e + len_e).  With
 * [x, y) its intersection with the ORF's [lo, hi): on '+' its forward interval is [cl + x - o_e, cl + y - o_e), on '-'
 * [ch - (y - o_e), ch - (x - o_e)); its GFF3 phase is (3 - (x - lo) mod 3) mod 3.  Segments the ORF does not touch (and
 * every segment of a record without an ORF) are reported empty: lo = hi = phase = -1.                                   */
#define MG_PRED_5PARTIAL 1
#define MG_PRED_3PARTIAL 2
typedef struct {
    int64_t lo, hi;               /* ORF in S, [lo, hi), stop included; -1, -1 = none                        */
    int32_t n_aa;                 /* residues, stop excluded; 0 = none                                       */
    int8_t  frame;                /* lo mod 3                                                                */
    int8_t  type;                 /* bit 0: 5' partial, bit 1: 3' partial                                    */
    uint8_t start_codon;          /* codon at lo, 16*b0+4*b1+b2; 0xFF = none or ambiguous                    */
    uint8_t stop_codon;           /* codon at hi-3 when there is a stop, else 0xFF                           */
    int32_t n_cds_seg;            /* caller segments the ORF touches                                         */
    int32_t pad;
} mg_cds_pred;                    /* 32 bytes */
typedef struct { int64_t lo, hi; int8_t phase; int8_t pad[7]; } mg_cds_seg;   /* 0-based half-open forward coords; -1,-1,-1 = empty */
/* rec_out[n_rec]; seg_out[n_seg] (one entry per caller segment, may be NULL).  flags: MG_PRED_5PARTIAL | MG_PRED_3PARTIAL.
 * Rules of mg_plan_check: a prepared plan on the genome as it is (MG_ESTATE otherwise; MG_PROT_DEFER is enough), the stop set
 * and the start set passed to the kernels by value.  mg_plan_predict_cds takes host outputs and copies them in stream order
 * (sync before reading; its device scratch grows outside a capture only); mg_plan_predict_cds_device takes device outputs and
 * queues two launches on `stream` with no host round trip, so a CUDA graph can capture it.                                */
int mg_plan_predict_cds(mg_plan *p, int64_t min_aa, const uint8_t *start64, int flags,
                        mg_cds_pred *rec_out, mg_cds_seg *seg_out, void *stream);
int mg_plan_predict_cds_device(mg_plan *p, int64_t min_aa, const uint8_t *start64, int flags,
                               mg_cds_pred *rec_out, mg_cds_seg *seg_out, void *stream);

/* ---- host side: native GFF3 / GTF reader + flattener (no GPU work; csrc/mg_gff.cu) ------------------------------------------
 * mg_gff_parse replaces read_gff (genome.py:242-415: line filter, version detection, attribute parsing, ID naming, de-dup,
 * implicit parents, child lists) on interned integer ids; `opts` is the option blob magot_b200/gffnative.py packs (format
 * version, features_to_ignore, base_features, parents_hierarchy, features_to_replace, IDfield, parent_field, and the tables /
 * objects an existing AnnotationSet already holds).  `text` must stay alive while the handle lives.  mg_gff_info: [0] status
 * (0 ok; else the line the reference stops at: 1 GFF2 attribute without value, 2 parent without a line, 3 GFF3 attribute
 * without '=', 4 bad coordinate, ...), [3] rows, [4] strings, ...  mg_gff_column / mg_gff_strings / mg_gff_find expose the SoA
 * columns (ids, coords, strand, phase, attributes, child lists, tables in dict insertion order) and the string table.
 * mg_gff_flatten replaces AnnotationSet.get_fasta / ParentAnnotation.get_fasta's choice of children, order and header
 * (genome.py:578-582, :683-719) for the rows `tops` of one feature table: it emits the arrays mg_plan_create takes.           */
typedef struct mg_gff mg_gff;
typedef struct mg_gff_flat mg_gff_flat;
int mg_gff_parse(const uint8_t *text, int64_t n, const uint8_t *opts, int64_t n_opts, mg_gff **out);
int mg_gff_destroy(mg_gff *m);
int mg_gff_info(mg_gff *m, int64_t *info16);
int mg_gff_column(mg_gff *m, const char *name, const void **ptr, int64_t *n, int32_t *elem_size);
int mg_gff_strings(mg_gff *m, const int32_t *ids, int64_t n, uint8_t *pool, int64_t cap, int64_t *off);
int64_t mg_gff_find(mg_gff *m, const uint8_t *s, int64_t n);
/* Iteration order of a CPython-2.7 dict holding the n keys pool[off[i], off[i+1]) inserted in that order (the reference prints
 * records by iterating plain dicts, genome.py:580, genome_tools.py:385; rounds = 2: after read_gff's copy.deepcopy, genome.py:415).
 * perm[k] = input index of the k-th key yielded.  mg_gff_py2_order: the same on string ids of a model.  Host only.            */
int mg_py2_order(const uint8_t *pool, const int64_t *off, int64_t n, int rounds, int64_t *perm);
int mg_gff_py2_order(mg_gff *m, const int32_t *ids, int64_t n, int rounds, int64_t *perm);
int mg_gff_flatten(mg_gff *m, const int64_t *tops, int64_t n_top, const int32_t *contig_of, int64_t n_contig_of, int framing,
                   mg_gff_flat **out);
int mg_gff_flat_destroy(mg_gff_flat *f);
int mg_gff_flat_column(mg_gff_flat *f, const char *name, const void **ptr, int64_t *n, int32_t *elem_size);

/* ---- timing / sync helpers ----------------------------------------------------------------- */
int mg_stream_sync(int device, void *stream);
/* Stream-ordered copy of n bytes from a device buffer (e.g. the output of an mg_emit_*_device call) to host memory (pinned
 * for full PCIe speed): the output side of `print annotation_set.get_fasta(...)` (genome_tools.py:324-330) when the caller
 * places the texts of several shards / GPUs in one host buffer itself.                                                */
int mg_copy_d2h_async(int device, void *dst_host, const void *src_dev, int64_t n, void *stream);
/* CUDA graphs: capture everything queued on `stream` (and on streams joined to it with mg_stream_wait_stream) between
 * mg_graph_begin and mg_graph_end -- e.g. mg_plan_prepare_async + mg_emit_*_device of several plans, none of which waits for
 * the host -- and replay it with one launch.  The batch-level counterpart of the reference's per-object loop
 * `for obj in table: obj.get_fasta()` (genome.py:578-582).  Buffers and plan handles used inside must stay alive and unchanged
 * in size while the graph is in use.  A capture needs the plan's buffers to exist already: run mg_plan_prepare_async (and
 * mg_emit_products_device) once outside the capture with at least the captured capacities; a call that would grow a buffer
 * inside a capture fails with MG_ESTATE before it queues anything.                                                      */
int mg_graph_begin(int device, void *stream);
int mg_graph_end(int device, void *stream, void **graph_exec_out);
int mg_graph_launch(int device, void *graph_exec, void *stream);
int mg_graph_destroy(void *graph_exec);
/* `waiter` waits for everything queued so far on `signaller` (event record + wait; usable inside a capture). */
int mg_stream_wait_stream(int device, void *waiter, void *signaller);
/* Developer / test knob: run-time choice between kernel variants that give bit-identical results ("emit": 0 = k_emit_nuc
 * (default), 1 = bulk-copy staged, 2 = streaming; "k1": 0 = piece-parallel plan launches (default), 1 = one-launch plan kernel;
 * "six": K4 scan for min_aa >= 96: 2 = two-level scan over the stop-codon index (default), 1 = two-level scan on the packed
 * bases, 0 = single-pass scan; "fuse": 1 = mg_emit_nuc_prot_* as one fused launch (default), 0 = as K2 + K3;
 * "multi_lag": distance between the products of mg_emit_products_device in millionths of a text).  */
int mg_tune(const char *key, int value);
/* Number of kernels launched by this library since load (per process), for bench accounting. */
int64_t mg_kernel_launches(void);

#ifdef __cplusplus
}
#endif
#endif /* MAGOT_B200_H */
