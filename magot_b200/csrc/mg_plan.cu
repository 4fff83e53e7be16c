// mg_plan.cu -- K1: SoA interval tables on the device, Python-slice clamping, piece table, prefix sums.
//
// A plan turns "n_rec records, each a list of segments in emission order + a literal prefix/suffix"
// into ONE flat piece table for the nucleotide text and ONE flat record table for the protein text:
//
//   piece p of record r:  F(r) = rec_seg_off[r] + 2r      -> literal prefix  (">ID\n")
//                         F(r)+1+k                          -> k-th segment   (genome interval, fwd or rc)
//                         F(r+1)-1                          -> literal suffix ("\n")
//   piece_off[p]  = byte offset of piece p in the nucleotide text (exclusive prefix sum of lengths)
//   piece_src[p]  = global base index of the lowest base of the interval (or offset into lit[]) | kind<<62
//
// so the emit kernels are flat, perfectly load-balanced passes over OUTPUT bytes (16 per thread), not
// over transcripts -- transcript lengths are heavy-tailed (188..8502 bp in the reference's own test set).
// Replaces the per-child bookkeeping of ParentAnnotation.get_fasta (genome.py:687-705) and the slice
// arithmetic of BaseAnnotation.get_seq (genome.py:603-608).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include "mg_common.cuh"
#include "mg_gather.cuh"
#include "mg_lookback.cuh"

// ---- kernels ----------------------------------------------------------------------------------------

#define PLAN_THREADS 256
#ifndef PLAN_ITEMS
#define PLAN_ITEMS 8                                 // pieces per thread of k_plan_pieces (a power of two >= 4)
#endif
#define PLAN_TILE (PLAN_THREADS * PLAN_ITEMS)        // pieces per block; 4096 (34 KB of shared memory) was faster alone but
                                                     // slowed the step by 0.06 ms: its blocks found no room next to K2
#define PLAN_WORDS (PLAN_TILE / 32)                  // words of the block's record-head bitmap

// thread per record: record r owns pieces [F(r), F(r+1)), F(r) = rec_seg_off[r] + 2r; it writes itself into every
// PLAN_TILE-piece block whose first piece it owns (coalesced and search-free; a binary search per block was 10 us of dependent loads)
__global__ void __launch_bounds__(256) k_plan_block_rec(int64_t n_block, int64_t n_rec, const int64_t *__restrict__ rec_seg_off,
                                                        int64_t *__restrict__ blk_r0) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const int64_t f0 = __ldg(rec_seg_off + r) + 2 * r, f1 = __ldg(rec_seg_off + r + 1) + 2 * (r + 1);
    for (int64_t b = (f0 + PLAN_TILE - 1) / PLAN_TILE; b * PLAN_TILE < f1 && b < n_block; b++) blk_r0[b] = r;
}

// tile -> first piece by scatter (mg_plan_prepare_async: the table exists before the text size is known): the piece that holds
// byte t * MG_NUC_TILE writes itself into slot t; the same at 1 KB granularity (one warp of k_emit_nuc_stream = one 1 KB block)
// when the streaming K2 asks for it.  Empty pieces hold no byte.
__device__ __forceinline__ void plan_scatter_nuc(int64_t off, int64_t len, int64_t p, int64_t *__restrict__ tile_first,
                                                 int64_t tile_cap, int32_t *__restrict__ blk1k, int64_t blk1k_cap) {
    if (len <= 0) return;
    if (tile_first)
        for (int64_t t = (off + MG_NUC_TILE - 1) / MG_NUC_TILE; t * MG_NUC_TILE < off + len && t < tile_cap; t++) tile_first[t] = p;
    for (int64_t t = (off + 1023) >> 10; (t << 10) < off + len && t < blk1k_cap; t++) blk1k[t] = (int32_t)p;
}

// K1 piece pass: clamp like a Python slice, write piece_src and -- through a block scan of the lengths plus a decoupled
// look-back across blocks (mg_lookback.cuh) -- every piece's offset in the nucleotide text, in one launch.
//   1. thread per record of the block: the two literal pieces (src, length) and a bit per record head in s_head;
//   2. thread per piece, strided so the segment tables are read coalesced: record = popcount of the heads up to the piece,
//      segment = piece - 2 * record - 1; literal pieces were written in 1, so the loop has one body;
//   3. a thread sums PLAN_ITEMS consecutive lengths, one block scan, one look-back;
//   4. the offsets go through shared memory (swizzled) back to the strided order: piece_off is written coalesced.
#ifndef PLAN_MINB
#define PLAN_MINB 6                                  // 40 registers, 17 KB of shared memory: no spill at 8 items (32 registers spill)
#endif
__global__ void __launch_bounds__(PLAN_THREADS, PLAN_MINB) k_plan_pieces(int64_t n_piece, int64_t n_rec, const int64_t *__restrict__ rec_seg_off,
                                                     const int64_t *__restrict__ blk_r0,
                                                     const int32_t *__restrict__ seg_contig, const int64_t *__restrict__ seg_start,
                                                     const int64_t *__restrict__ seg_end, const int8_t *__restrict__ seg_strand,
                                                     const int64_t *__restrict__ rec_lit_off, const int32_t *__restrict__ rec_pre,
                                                     const int32_t *__restrict__ rec_suf, const int64_t *__restrict__ contig_len,
                                                     const int64_t *__restrict__ contig_base, int64_t n_contigs, int64_t two_T,
                                                     unsigned long long *tmp, int64_t *__restrict__ piece_off,
                                                     int64_t *__restrict__ piece_src, int64_t *__restrict__ total_out,
                                                     int64_t *__restrict__ tile_first, int64_t tile_cap,
                                                     int32_t *__restrict__ blk1k, int64_t blk1k_cap) {
    // s_len (piece lengths: a piece is < 2^31 bytes) until step 3, then s_off (block-relative offsets, 64 bits)
    __shared__ __align__(16) int64_t s_buf[PLAN_TILE];
    uint32_t *s_len = reinterpret_cast<uint32_t *>(s_buf);
    __shared__ uint32_t s_head[PLAN_WORDS + 1];       // bit j: piece pb + j is a literal prefix (bit PLAN_TILE: the piece after the block)
    __shared__ uint32_t s_cnt[PLAN_WORDS];            // heads in the words before
    __shared__ int64_t s_warp[8];
    __shared__ int64_t s_prefix;
    __shared__ unsigned int s_tile;
    for (int i = threadIdx.x; i <= PLAN_WORDS; i += PLAN_THREADS) s_head[i] = 0;
    const int64_t tile = mg_next_tile(tmp, &s_tile);
    const int64_t pb = tile * PLAN_TILE;
    const int nt = (int)min((int64_t)PLAN_TILE, n_piece - pb);   // pieces of this block
    const int64_t pe = pb + nt;
    const int64_t r0 = blk_r0[tile];                 // the record that owns piece pb (k_plan_block_rec)

    // 1. Record r writes its prefix F(r) and suffix F(r+1)-1 where they fall in the block and marks F(r+1), the next record's
    // head; r0 marks its own head when it starts the block.  Rounds of PLAN_THREADS records until one ends at or past pe.
    for (int64_t r = r0 + threadIdx.x;; r += PLAN_THREADS) {
        bool more = false;
        if (r < n_rec) {
            const int64_t f0 = __ldg(rec_seg_off + r) + 2 * r;
            if (f0 < pe) {
                const int64_t f1 = __ldg(rec_seg_off + r + 1) + 2 * (r + 1);
                const int64_t lit = __ldg(rec_lit_off + r);
                const int32_t pre = __ldg(rec_pre + r), suf = __ldg(rec_suf + r);
                if (f0 >= pb) {
                    s_len[f0 - pb] = (uint32_t)pre;
                    piece_src[f0] = lit | (int64_t)(MG_KIND_LIT << MG_KIND_SHIFT);
                    if (f0 == pb) atomicOr(&s_head[0], 1u);
                }
                if (f1 - 1 < pe) {
                    s_len[f1 - 1 - pb] = (uint32_t)suf;
                    piece_src[f1 - 1] = (lit + pre) | (int64_t)(MG_KIND_LIT << MG_KIND_SHIFT);
                }
                if (f1 - pb <= PLAN_TILE) atomicOr(&s_head[(f1 - pb) >> 5], 1u << ((f1 - pb) & 31));
                more = f1 < pe;
            }
        }
        if (!__syncthreads_and(more)) break;         // records grow with the thread index: the round's last one decides
    }
    if (threadIdx.x < 32) {                          // heads before each word: one warp, PLAN_WORDS / 32 words a lane
        uint32_t c[PLAN_WORDS / 32], sum = 0;
#pragma unroll
        for (int k = 0; k < PLAN_WORDS / 32; k++) { c[k] = __popc(s_head[threadIdx.x * (PLAN_WORDS / 32) + k]); sum += c[k]; }
        uint32_t incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)threadIdx.x >= d) incl += t;
        }
        uint32_t run = incl - sum;
#pragma unroll
        for (int k = 0; k < PLAN_WORDS / 32; k++) { s_cnt[threadIdx.x * (PLAN_WORDS / 32) + k] = run; run += c[k]; }
    }
    __syncthreads();

    // 2. Genome segments.  A warp's 32 pieces of one round are one word of s_head, so lane l's record is r0 plus the heads in
    // bits 0..l (less one when the block starts with r0's own prefix).
    const int lane = threadIdx.x & 31;
    const uint32_t upto = 0xffffffffu >> (31 - lane);
    const int64_t rb = r0 - (int64_t)(s_head[0] & 1u);
#pragma unroll 4
    for (int it = 0; it < PLAN_ITEMS; it++) {
        const int j = it * PLAN_THREADS + threadIdx.x, w = j >> 5;
        if (j >= nt) { s_len[j] = 0; continue; }
        const uint32_t h = s_head[w];
        const uint32_t lit = h | (h >> 1) | (s_head[w + 1] << 31);   // a head (prefix) or the piece before one (suffix)
        if ((lit >> lane) & 1u) continue;
        const int64_t p = pb + j;
        const int64_t e = p - 2 * (rb + s_cnt[w] + __popc(h & upto)) - 1;
        const int32_t c = __ldg(seg_contig + e);
        const int64_t s = __ldg(seg_start + e), en = __ldg(seg_end + e);
        const int8_t minus = __ldg(seg_strand + e);
        int64_t src = MG_FRONT_PAD, n = 0;
        if (c >= 0 && c < n_contigs) {
            const int64_t L = __ldg(contig_len + c);
            // contig[start-1:end] with Python slice semantics (genome.py:606)
            int64_t i = s - 1, k = en;
            if (i < 0) { i += L; if (i < 0) i = 0; } else if (i > L) i = L;
            if (k < 0) { k += L; if (k < 0) k = 0; } else if (k > L) k = L;
            n = k > i ? k - i : 0;
            if (n > 0x7fffffff) n = 0x7fffffff;   // not reached: mg_plan_create splits longer segments
            src = __ldg(contig_base + c) + i;
        }
        s_len[j] = (uint32_t)n;
        // '-' strand: forward bases [src, src+len) are bases [2T-src-len, 2T-src) of the reverse-complement plane,
        // in exactly the order Sequence.reverse_compliment emits them (genome.py:784-793)
        piece_src[p] = minus ? two_T - src - n : src;
    }
    __syncthreads();

    // 3. blocked: a thread owns PLAN_ITEMS consecutive pieces, so the block needs ONE scan
    uint32_t len[PLAN_ITEMS];
    int64_t mine = 0;
#pragma unroll
    for (int q = 0; q < PLAN_ITEMS / 4; q++) {
        const uint4 u = reinterpret_cast<const uint4 *>(s_len + threadIdx.x * PLAN_ITEMS)[q];
        len[4 * q] = u.x; len[4 * q + 1] = u.y; len[4 * q + 2] = u.z; len[4 * q + 3] = u.w;
        mine += (int64_t)u.x + (int64_t)u.y + (int64_t)u.z + (int64_t)u.w;
    }
    int64_t total;
    const int64_t incl = mg_block_incl_scan(mine, s_warp, &total);   // its barriers also end every read of s_len
    int64_t run = incl - mine;
#pragma unroll
    for (int i = 0; i < PLAN_ITEMS; i++) {           // slot rotated by the thread index: two wavefronts a warp store
        s_buf[threadIdx.x * PLAN_ITEMS + ((i + threadIdx.x) & (PLAN_ITEMS - 1))] = run;
        run += len[i];
    }
    const int64_t prefix = mg_lookback(tmp, tile, total, &s_prefix);   // ends with a barrier

    // 4. strided again: coalesced piece_off, and the tile tables
#pragma unroll 4
    for (int it = 0; it < PLAN_ITEMS; it++) {
        const int j = it * PLAN_THREADS + threadIdx.x;
        if (j >= nt) break;
        const int t0 = j / PLAN_ITEMS, t1 = (j + 1) / PLAN_ITEMS;
        const int64_t o0 = s_buf[t0 * PLAN_ITEMS + ((j + t0) & (PLAN_ITEMS - 1))];
        const int64_t o1 = j + 1 < nt ? s_buf[t1 * PLAN_ITEMS + ((j + 1 + t1) & (PLAN_ITEMS - 1))] : total;
        const int64_t off = prefix + o0;
        piece_off[pb + j] = off;
        plan_scatter_nuc(off, o1 - o0, pb + j, tile_first, tile_cap, blk1k, blk1k_cap);
    }
    if (tile == gridDim.x - 1 && threadIdx.x == 0) {
        const int64_t all = prefix + total;
        piece_off[n_piece] = all;
        *total_out = all;
        if (tile_first) {                              // sentinel after the last tile, as k_plan_tiles writes it
            const int64_t n_tile = min(tile_cap, (all + MG_NUC_TILE - 1) / MG_NUC_TILE);
            tile_first[n_tile] = n_piece > 0 ? n_piece - 1 : 0;
        }
        const int64_t n_blk = (all + 1023) >> 10;
        if (n_blk < blk1k_cap) blk1k[n_blk] = (int32_t)(n_piece > 0 ? n_piece - 1 : 0);
    }
}

// K1 record pass: spliced length -> amino-acid count (Sequence.translate, genome.py:810-821) and, with a block scan + look-back,
// the record's offset in the protein text.  A thread owns REC_ITEMS consecutive records, and a record costs three dependent
// trips in the common case: its rec_seg_off words; the offsets of its prefix, first two segment pieces, suffix and the first
// segment's source; the first codon, read straight from that segment when it holds skip + 3 bases.
#define REC_THREADS 256
#ifndef REC_ITEMS
#define REC_ITEMS 2                                  // 4 was slower at 1/8 of config 4 (fewer blocks in flight)
#endif
#define REC_TILE (REC_THREADS * REC_ITEMS)
__global__ void __launch_bounds__(REC_THREADS) k_plan_records(int64_t n_rec, const int64_t *__restrict__ rec_seg_off,
                                                      const int64_t *__restrict__ piece_off, const int64_t *__restrict__ piece_src,
                                                      const uint32_t *__restrict__ packed, const int8_t *__restrict__ rec_phase,
                                                      int flags, int32_t *__restrict__ rec_aa, int8_t *__restrict__ rec_skip,
                                                      unsigned long long *tmp, int64_t *__restrict__ prot_off,
                                                      int64_t *__restrict__ total_out, int64_t *__restrict__ tile_first,
                                                      int64_t tile_cap) {
    __shared__ int64_t s_warp[8];
    __shared__ int64_t s_prefix;
    __shared__ unsigned int s_tile;
    const int64_t tile = mg_next_tile(tmp, &s_tile);
    const int64_t r0 = tile * REC_TILE + (int64_t)threadIdx.x * REC_ITEMS;
    const bool phase = (flags & MG_PROT_USE_PHASE) && rec_phase;
    int64_t so[REC_ITEMS + 1];
    int ph[REC_ITEMS];
#pragma unroll
    for (int k = 0; k <= REC_ITEMS; k++) so[k] = r0 + k <= n_rec ? __ldg(rec_seg_off + r0 + k) : 0;
#pragma unroll
    for (int k = 0; k < REC_ITEMS; k++) ph[k] = phase && r0 + k < n_rec ? rec_phase[r0 + k] : 0;
    int64_t plen[REC_ITEMS], mine = 0;
#pragma unroll
    for (int k = 0; k < REC_ITEMS; k++) {
        const int64_t r = r0 + k;
        plen[k] = 0;
        if (r >= n_rec) continue;
        const int64_t f0 = so[k] + 2 * r, f1 = so[k + 1] + 2 * (r + 1);
        // f0 + 2 <= f1 <= n_piece: all five offsets exist; piece f0 + 1 is the first segment whenever the payload is not empty
        const int64_t o_pre = __ldg(piece_off + f0), pay0 = __ldg(piece_off + f0 + 1), o_2 = __ldg(piece_off + f0 + 2);
        const int64_t pay1 = __ldg(piece_off + f1 - 1), o_end = __ldg(piece_off + f1);
        const int64_t src1 = __ldg(piece_src + f0 + 1) & (int64_t)MG_SRC_MASK;
        int skip = ph[k];
        if (skip < 0 || skip > 2) skip = 0;
        const int64_t L = pay1 - pay0 - skip;
        int64_t naa;
        if (L <= 2) {
            naa = -1;                                    // reference returns None (genome.py:810)
        } else {
            naa = L / 3;
            if (flags & MG_PROT_TRIMX) {                 // drop exactly one leading X (genome.py:819-821)
                const int64_t S = pay0 + skip;
                uint32_t n3;
                if (S + 3 <= o_2) {
                    n3 = (uint32_t)mg_ld_nib16(packed, src1 + skip);
                } else {                                 // the codon starts past, or runs out of, the first segment: walk
                    uint64_t acc[3];
                    int64_t j = f0 + 1;
                    while (j + 1 < f1 - 1 && __ldg(piece_off + j + 1) <= S) j++;
                    mg_gather_nib(packed, piece_off, piece_src, j, S, 3, acc);
                    n3 = (uint32_t)acc[0];
                }
                if (n3 & 0x888u) { naa -= 1; skip += 3; }
            }
        }
        if (naa > 0x7fffffff) naa = 0x7fffffff;
        rec_aa[r] = (int32_t)naa;
        rec_skip[r] = (int8_t)skip;
        plen[k] = (pay0 - o_pre) + (naa > 0 ? naa : 0) + (o_end - pay1);
        mine += plen[k];
    }
    int64_t total;
    const int64_t incl = mg_block_incl_scan(mine, s_warp, &total);
    const int64_t prefix = mg_lookback(tmp, tile, total, &s_prefix);
    int64_t off = prefix + incl - mine;
#pragma unroll
    for (int k = 0; k < REC_ITEMS; k++) {
        const int64_t r = r0 + k;
        if (r >= n_rec) break;
        prot_off[r] = off;
        if (tile_first && plen[k] > 0) {               // tile -> first record by scatter, see plan_scatter_nuc
            for (int64_t t = (off + MG_PROT_TILE - 1) / MG_PROT_TILE; t * MG_PROT_TILE < off + plen[k] && t < tile_cap; t++) tile_first[t] = r;
        }
        off += plen[k];
    }
    if (tile == gridDim.x - 1 && threadIdx.x == 0) {
        const int64_t all = prefix + total;
        prot_off[n_rec] = all;
        *total_out = all;
        if (tile_first) {
            const int64_t n_tile = min(tile_cap, (all + MG_PROT_TILE - 1) / MG_PROT_TILE);
            tile_first[n_tile] = n_rec > 0 ? n_rec - 1 : 0;
        }
    }
}


// ---- K1 in ONE kernel: thread per record ---------------------------------------------------------------------------------
// Round 1 ran K1 as a memset + three dependent launches (record of every 1024-piece block, thread per piece, thread per
// record): 65-85 us of mostly launch and load latency that does not shrink with the batch (37 us for 1/8 of config 4: the
// limiter of strong scaling, SCALE_r01 / bench line r2g).  Here a thread walks the segments of its record twice: pass 1 clamps
// (Python slice rules, genome.py:606), sums the payload and picks up the first codon for trimX (genome.py:819-821); two block
// scans + decoupled look-backs give the record's offsets in the nucleotide and the protein text; pass 2 writes the piece
// table and the tile / 1 KB block tables.  No record search, no staging, one launch.  A record's pieces are contiguous, so a
// thread writes a contiguous run of both tables.  Used when no record has more than PR_MAXSEG segments (the slowest thread
// bounds the kernel); else the piece-parallel kernels above.
#define PR_THREADS 256
#ifndef PR_MAXSEG
#define PR_MAXSEG 256
#endif

struct pr_seg { int64_t src; int64_t n; };             // piece source (plane index of its first emitted base) and clamped length

__device__ __forceinline__ pr_seg pr_clamp(int64_t e, const int32_t *__restrict__ seg_contig, const int64_t *__restrict__ seg_start,
                                           const int64_t *__restrict__ seg_end, const int8_t *__restrict__ seg_strand,
                                           const int64_t *__restrict__ contig_len, const int64_t *__restrict__ contig_base,
                                           int64_t n_contigs, int64_t two_T) {
    const int32_t c = __ldg(seg_contig + e);
    int64_t src = MG_FRONT_PAD, n = 0;
    if (c >= 0 && c < n_contigs) {
        const int64_t L = __ldg(contig_len + c);
        // contig[start-1:end] with Python slice semantics (genome.py:606)
        int64_t i = __ldg(seg_start + e) - 1, j = __ldg(seg_end + e);
        if (i < 0) { i += L; if (i < 0) i = 0; } else if (i > L) i = L;
        if (j < 0) { j += L; if (j < 0) j = 0; } else if (j > L) j = L;
        n = j > i ? j - i : 0;
        if (n > 0x7fffffff) n = 0x7fffffff;       // not reached: mg_plan_create splits longer segments
        src = __ldg(contig_base + c) + i;
    }
    // '-' strand: forward bases [src, src+n) are bases [2T-src-n, 2T-src) of the reverse-complement plane, in the order
    // Sequence.reverse_compliment emits them (genome.py:784-793)
    pr_seg r;
    r.src = __ldg(seg_strand + e) ? two_T - src - n : src;
    r.n = n;
    return r;
}

__device__ __forceinline__ void pr_scatter(int64_t off, int64_t len, int64_t p, int64_t *__restrict__ tile_first, int64_t tile_cap,
                                           int32_t *__restrict__ blk1k, int64_t blk1k_cap) {
    if (len <= 0) return;
    if (tile_first)
        for (int64_t t = (off + MG_NUC_TILE - 1) / MG_NUC_TILE; t * MG_NUC_TILE < off + len && t < tile_cap; t++) tile_first[t] = p;
    for (int64_t t = (off + 1023) >> 10; (t << 10) < off + len && t < blk1k_cap; t++) blk1k[t] = (int32_t)p;
}

#define PR_RECS 128                                   // records per block (threads 0..127 own one each)
#ifndef PR_SEGCAP
#define PR_SEGCAP 3072                                // clamped segments staged per block (config 4: ~1500); the rest is re-clamped from global memory
#endif

__global__ void __launch_bounds__(PR_THREADS) k_plan_rec(
    int64_t n_rec, int64_t n_piece, const int64_t *__restrict__ rec_seg_off, const int32_t *__restrict__ seg_contig,
    const int64_t *__restrict__ seg_start, const int64_t *__restrict__ seg_end, const int8_t *__restrict__ seg_strand,
    const int64_t *__restrict__ rec_lit_off, const int32_t *__restrict__ rec_pre, const int32_t *__restrict__ rec_suf,
    const int8_t *__restrict__ rec_phase, int flags, const int64_t *__restrict__ contig_len, const int64_t *__restrict__ contig_base,
    int64_t n_contigs, int64_t two_T, const uint32_t *__restrict__ packed, unsigned long long *tmp_a, unsigned long long *tmp_b,
    int64_t *__restrict__ piece_off, int64_t *__restrict__ piece_src, int64_t *__restrict__ prot_off, int32_t *__restrict__ rec_aa,
    int8_t *__restrict__ rec_skip, int64_t *__restrict__ totals, int64_t *__restrict__ tf_nuc, int64_t cap_nuc,
    int64_t *__restrict__ tf_prot, int64_t cap_prot, int32_t *__restrict__ blk1k, int64_t blk1k_cap) {
    // Phase 1 (all threads, parallel over the block's segments, coalesced): clamp every segment once into shared memory.
    // Phase 2 (thread per record, serial over ITS segments in shared memory): payload length, first codon, protein length.
    // Phase 3: block scans + look-backs.  Phase 4 (thread per record): piece table, tile tables.
    __shared__ int64_t s_src[PR_SEGCAP];
    __shared__ int32_t s_n[PR_SEGCAP];
    __shared__ int64_t s_warp[8];
    __shared__ int64_t s_prefix;
    __shared__ unsigned int s_tile;
    const int64_t tile = mg_next_tile(tmp_a, &s_tile);
    const int64_t r_first = tile * PR_RECS;
    const int64_t r_last = min(r_first + PR_RECS, n_rec);
    const int64_t e_lo = __ldg(rec_seg_off + r_first), e_hi = __ldg(rec_seg_off + r_last);
    const int n_stage = (int)min(e_hi - e_lo, (int64_t)PR_SEGCAP);
#pragma unroll 4
    for (int i = threadIdx.x; i < n_stage; i += PR_THREADS) {
        const pr_seg sg = pr_clamp(e_lo + i, seg_contig, seg_start, seg_end, seg_strand, contig_len, contig_base, n_contigs, two_T);
        s_src[i] = sg.src;
        s_n[i] = (int32_t)sg.n;
    }
    __syncthreads();
    const int64_t r = r_first + threadIdx.x;
    const bool mine = threadIdx.x < PR_RECS && r < n_rec;
    int64_t s0 = 0, s1 = 0, L = 0, lit = 0;
    int pre = 0, suf = 0;
    int64_t naa = 0;
    int skip = 0;
    if (mine) {
        s0 = __ldg(rec_seg_off + r);
        s1 = __ldg(rec_seg_off + r + 1);
        pre = rec_pre[r];
        suf = rec_suf[r];
        lit = rec_lit_off[r];
        if ((flags & MG_PROT_USE_PHASE) && rec_phase) { skip = rec_phase[r]; if (skip < 0 || skip > 2) skip = 0; }
        uint32_t first = 0;                              // the first five spliced bases (a codon after a phase of 0..2)
        int got = 0;
        for (int64_t e = s0; e < s1; e++) {
            pr_seg sg;
            const int64_t i = e - e_lo;
            if (i < n_stage) { sg.src = s_src[i]; sg.n = s_n[i]; }
            else sg = pr_clamp(e, seg_contig, seg_start, seg_end, seg_strand, contig_len, contig_base, n_contigs, two_T);
            if (got < 5 && sg.n > 0) {
                const int take = (int)min((int64_t)(5 - got), sg.n);
                const uint32_t v = (uint32_t)mg_ld_nib16(packed, sg.src) & ((1u << (4 * take)) - 1u);
                first |= v << (4 * got);
                got += take;
            }
            L += sg.n;
        }
        const int64_t Lp = L - skip;
        if (Lp <= 2) {
            naa = -1;                                    // reference returns None (genome.py:810)
        } else {
            naa = Lp / 3;
            if ((flags & MG_PROT_TRIMX) && (((first >> (4 * skip)) & 0xFFFu) & 0x888u)) { naa -= 1; skip += 3; }   // one leading X (genome.py:819-821)
        }
        if (naa > 0x7fffffff) naa = 0x7fffffff;
        rec_aa[r] = (int32_t)naa;
        rec_skip[r] = (int8_t)skip;
    }
    const int64_t nbytes = mine ? pre + L + suf : 0;
    const int64_t pbytes = mine ? pre + (naa > 0 ? naa : 0) + suf : 0;
    int64_t tot_n, tot_p;
    const int64_t incl_n = mg_block_incl_scan(nbytes, s_warp, &tot_n);
    const int64_t pre_n = mg_lookback(tmp_a, tile, tot_n, &s_prefix);
    const int64_t incl_p = mg_block_incl_scan(pbytes, s_warp, &tot_p);
    const int64_t pre_p = mg_lookback(tmp_b, tile, tot_p, &s_prefix);
    if (mine) {
        int64_t off = pre_n + incl_n - nbytes;
        int64_t p = s0 + 2 * r;
        piece_off[p] = off;
        piece_src[p] = lit | (int64_t)(MG_KIND_LIT << MG_KIND_SHIFT);
        pr_scatter(off, pre, p, tf_nuc, cap_nuc, blk1k, blk1k_cap);
        off += pre;
        p++;
        for (int64_t e = s0; e < s1; e++, p++) {
            pr_seg sg;
            const int64_t i = e - e_lo;
            if (i < n_stage) { sg.src = s_src[i]; sg.n = s_n[i]; }
            else sg = pr_clamp(e, seg_contig, seg_start, seg_end, seg_strand, contig_len, contig_base, n_contigs, two_T);
            piece_off[p] = off;
            piece_src[p] = sg.src;
            pr_scatter(off, sg.n, p, tf_nuc, cap_nuc, blk1k, blk1k_cap);
            off += sg.n;
        }
        piece_off[p] = off;
        piece_src[p] = (lit + pre) | (int64_t)(MG_KIND_LIT << MG_KIND_SHIFT);
        pr_scatter(off, suf, p, tf_nuc, cap_nuc, blk1k, blk1k_cap);
        const int64_t poff = pre_p + incl_p - pbytes;
        prot_off[r] = poff;
        if (tf_prot && pbytes > 0)
            for (int64_t t = (poff + MG_PROT_TILE - 1) / MG_PROT_TILE; t * MG_PROT_TILE < poff + pbytes && t < cap_prot; t++) tf_prot[t] = r;
    }
    if (tile == gridDim.x - 1 && threadIdx.x == 0) {
        const int64_t all_n = pre_n + tot_n, all_p = pre_p + tot_p;
        piece_off[n_piece] = all_n;
        prot_off[n_rec] = all_p;
        totals[0] = all_n;
        totals[1] = all_p;
        if (tf_nuc) tf_nuc[min(cap_nuc, (all_n + MG_NUC_TILE - 1) / MG_NUC_TILE)] = n_piece > 0 ? n_piece - 1 : 0;
        if (tf_prot) tf_prot[min(cap_prot, (all_p + MG_PROT_TILE - 1) / MG_PROT_TILE)] = n_rec > 0 ? n_rec - 1 : 0;
        const int64_t n_blk = (all_n + 1023) >> 10;
        if (n_blk < blk1k_cap) blk1k[n_blk] = (int32_t)(n_piece > 0 ? n_piece - 1 : 0);
    }
}

// thread per tile: index of the piece / record that contains the tile's first byte; nucleotide tiles first, then protein
// tiles.  The tile counts come from the totals ON THE DEVICE, so the launch needs no host round trip: the grid covers
// cap_a + cap_b + 2 slots (capacities of the two tables), threads beyond the real counts do nothing.
__global__ void __launch_bounds__(256) k_plan_tiles(const int64_t *__restrict__ totals, const int64_t *__restrict__ off_a, int64_t n_a,
                                                    int64_t tile_a, int64_t cap_a, int64_t *__restrict__ first_a,
                                                    const int64_t *__restrict__ off_b, int64_t n_b, int64_t tile_b, int64_t cap_b,
                                                    int64_t *__restrict__ first_b) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t *off = off_a;
    int64_t n = n_a, tile_bytes = tile_a, cap = cap_a, total = totals[0], *tile_first = first_a;
    if (t > cap_a) { t -= cap_a + 1; off = off_b; n = n_b; tile_bytes = tile_b; cap = cap_b; total = totals[1]; tile_first = first_b; }
    const int64_t n_tile = min(cap, (total + tile_bytes - 1) / tile_bytes);
    if (t > n_tile || n_tile == 0) return;
    if (t == n_tile) { tile_first[t] = n > 0 ? n - 1 : 0; return; }
    tile_first[t] = mg_search_le(off, 0, n, t * tile_bytes);
}

__global__ void __launch_bounds__(256) k_plan_lengths(int64_t n_rec, const int64_t *__restrict__ rec_seg_off,
                                                      const int64_t *__restrict__ piece_off, const int32_t *__restrict__ rec_aa,
                                                      int64_t *__restrict__ nuc_len, int64_t *__restrict__ aa_len) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const int64_t f0 = rec_seg_off[r] + 2 * r, f1 = rec_seg_off[r + 1] + 2 * (r + 1);
    if (nuc_len) nuc_len[r] = piece_off[f1 - 1] - piece_off[f0 + 1];
    if (aa_len) aa_len[r] = rec_aa[r];
}

// ---- host side ------------------------------------------------------------------------------------------
// K1 variant: env MAGOT_K1 or mg_tune("k1", v): 0 (default) = the three piece-parallel launches; 1 = k_plan_rec, one launch
// (measured on config 4: 0.105 / 0.121 ms per plan against 0.077 / 0.085 ms -- kept as a tested variant, not the default)
static int g_k1_mode = -1;
static int mg_k1_mode() {
    if (g_k1_mode < 0) {
        const char *e = getenv("MAGOT_K1");
        g_k1_mode = (e && !strcmp(e, "rec")) ? 1 : 0;
    }
    return g_k1_mode;
}
void mg_set_k1_mode(int v) { g_k1_mode = v ? 1 : 0; }

template <typename T>
static int upload(mg_plan *p, T **dst, const T *src, int64_t n, cudaStream_t st) {
    void *d = nullptr;
    MG_CUDA(cudaMallocAsync(&d, std::max<int64_t>(1, n) * sizeof(T), st));
    p->owned.push_back(d);
    if (n > 0 && src) MG_CUDA(cudaMemcpyAsync(d, src, n * sizeof(T), cudaMemcpyHostToDevice, st));
    *dst = (T *)d;
    return MG_OK;
}

template <typename T>
static int dalloc(mg_plan *p, T **dst, int64_t n, cudaStream_t st) {
    void *d = nullptr;
    MG_CUDA(cudaMallocAsync(&d, std::max<int64_t>(1, n) * sizeof(T), st));
    p->owned.push_back(d);
    *dst = (T *)d;
    return MG_OK;
}

extern "C" int mg_plan_create(mg_genome *g, int64_t n_rec, const int64_t *rec_seg_off, int64_t n_seg,
                              const int32_t *seg_contig, const int64_t *seg_start, const int64_t *seg_end,
                              const int8_t *seg_strand, const int64_t *rec_lit_off, const int32_t *rec_pre_len,
                              const int32_t *rec_suf_len, const uint8_t *lit, int64_t n_lit, const int8_t *rec_phase,
                              void *stream, mg_plan **out) {
    MG_REQUIRE(g != nullptr && out != nullptr, "NULL handle");
    MG_REQUIRE(g->finalized, "mg_genome_finalize has not been called");
    MG_REQUIRE(n_rec >= 0 && n_seg >= 0 && n_lit >= 0, "negative size");
    MG_REQUIRE(rec_seg_off != nullptr, "rec_seg_off is NULL");
    MG_REQUIRE(n_seg == 0 || (seg_contig && seg_start && seg_end && seg_strand), "segment arrays are NULL");
    MG_REQUIRE(n_rec == 0 || (rec_lit_off && rec_pre_len && rec_suf_len), "record arrays are NULL");
    MG_REQUIRE(rec_seg_off[0] == 0 && rec_seg_off[n_rec] == n_seg, "rec_seg_off must start at 0 and end at n_seg");
    // The Python-slice clamp of every segment (the rule of the plan kernels, genome.py:606), exactly, on the host: the nucleotide
    // text size, the protein limit of each record, and the segments the kernels cannot take as one piece.
    const int64_t SPLIT_AT = 1ll << 31, CHUNK = 1ll << 30;
    const int64_t REC_MAX = 3 * 0x7fffffffll + 2;     // rec_aa is int32: at most 2^31 - 1 amino acids of 3 bases each
    auto clamp = [&](int64_t e, int64_t *lo) -> int64_t {   // clamped length of segment e; *lo = its first base in the contig
        const int32_t c = seg_contig[e];
        *lo = 0;
        if (c < 0 || c >= g->n_contigs) return 0;
        const int64_t L = g->h_contig_len[c];
        int64_t i = seg_start[e] - 1, k = seg_end[e];
        if (i < 0) { i += L; if (i < 0) i = 0; } else if (i > L) i = L;
        if (k < 0) { k += L; if (k < 0) k = 0; } else if (k > L) k = L;
        *lo = i;
        return k > i ? k - i : 0;
    };
    int64_t nuc_bytes = 0;
    bool any_long = false;
    for (int64_t r = 0; r < n_rec; r++) {
        int64_t pay = 0, lo;
        for (int64_t e = rec_seg_off[r]; e < rec_seg_off[r + 1]; e++) {
            const int64_t n = clamp(e, &lo);
            any_long |= n >= SPLIT_AT;
            pay += n;
        }
        if (pay > REC_MAX) {
            mg_set_error("record %lld holds %lld bases: a record's payload is limited to 3 * (2^31 - 1) + 2 = %lld bases "
                         "(its protein length is an int32)", (long long)r, (long long)pay, (long long)REC_MAX);
            return MG_EINVAL;
        }
        nuc_bytes += pay + rec_pre_len[r] + rec_suf_len[r];
    }
    // Pieces are int32-long in the plan and emit kernels (piece lengths in shared memory, tile-relative offsets), so a segment of
    // 2^31 bases or more is split into consecutive chunks of at most 2^30 bases.  Each chunk lies inside its contig, so the
    // kernels' clamp leaves it alone; on '-' the chunks run from the slice's end to its start, because rc(s) = rc(last chunk) +
    // ... + rc(first chunk).  A table without such a segment is uploaded as it is.
    std::vector<int64_t> x_rec_seg_off, x_start, x_end;
    std::vector<int32_t> x_contig;
    std::vector<int8_t> x_strand;
    const int64_t n_cseg = n_seg;                     // the caller's table (mg_plan_check reports junctions per caller segment)
    const int64_t *c_rec_seg_off = rec_seg_off, *c_start = seg_start, *c_end = seg_end;
    const int32_t *c_contig = seg_contig;
    const int8_t *c_strand = seg_strand;
    if (any_long) {
        x_rec_seg_off.reserve(n_rec + 1);
        x_rec_seg_off.push_back(0);
        for (int64_t r = 0; r < n_rec; r++) {
            for (int64_t e = rec_seg_off[r]; e < rec_seg_off[r + 1]; e++) {
                int64_t lo0;
                const int64_t n = clamp(e, &lo0);
                if (n < SPLIT_AT) {
                    x_contig.push_back(seg_contig[e]); x_start.push_back(seg_start[e]); x_end.push_back(seg_end[e]);
                    x_strand.push_back(seg_strand[e]);
                    continue;
                }
                const int64_t k = (n + CHUNK - 1) / CHUNK;
                for (int64_t q = 0; q < k; q++) {
                    const int64_t j = seg_strand[e] ? k - 1 - q : q;
                    const int64_t lo = lo0 + j * CHUNK, hi = std::min(lo0 + n, lo + CHUNK);
                    x_contig.push_back(seg_contig[e]); x_start.push_back(lo + 1); x_end.push_back(hi);
                    x_strand.push_back(seg_strand[e]);
                }
            }
            x_rec_seg_off.push_back((int64_t)x_contig.size());
        }
        n_seg = (int64_t)x_contig.size();
        rec_seg_off = x_rec_seg_off.data();
        seg_contig = x_contig.data();
        seg_start = x_start.data();
        seg_end = x_end.data();
        seg_strand = x_strand.data();
    }
    MG_REQUIRE(n_seg + 2 * n_rec < 0x7fffffff, "more than 2^31 pieces in one plan: split the table");
    MG_CUDA(cudaSetDevice(g->device));
    cudaStream_t st = (cudaStream_t)stream;
    mg_plan *p = new mg_plan();
    p->g = g;
    p->device = g->device;
    p->n_rec = n_rec;
    p->n_seg = n_seg;
    p->n_piece = n_seg + 2 * n_rec;
    p->n_lit = n_lit;
    p->last_stream = st;
    int rc = MG_OK;
#define TRY(x) do { rc = (x); if (rc) { mg_plan_destroy(p); return rc; } } while (0)
    TRY(upload(p, &p->d_rec_seg_off, rec_seg_off, n_rec + 1, st));
    TRY(upload(p, &p->d_seg_contig, seg_contig, n_seg, st));
    TRY(upload(p, &p->d_seg_start, seg_start, n_seg, st));
    TRY(upload(p, &p->d_seg_end, seg_end, n_seg, st));
    TRY(upload(p, &p->d_seg_strand, seg_strand, n_seg, st));
    TRY(upload(p, &p->d_rec_lit_off, rec_lit_off, n_rec, st));
    TRY(upload(p, &p->d_rec_pre, rec_pre_len, n_rec, st));
    TRY(upload(p, &p->d_rec_suf, rec_suf_len, n_rec, st));
    {   // literal bytes sit 64 bytes into a zeroed, padded buffer: the emit kernels fetch 32-byte windows (as aligned
        // words) that may start up to 35 bytes before / end up to 39 bytes after the literal they need
        uint8_t *d = nullptr;
        TRY(dalloc(p, &d, n_lit + 128, st));
        rc = cudaMemsetAsync(d, 0, n_lit + 128, st) == cudaSuccess ? MG_OK : MG_ECUDA;
        if (rc == MG_OK && n_lit > 0 && cudaMemcpyAsync(d + 64, lit, n_lit, cudaMemcpyHostToDevice, st) != cudaSuccess) rc = MG_ECUDA;
        if (rc) { mg_set_error("literal upload failed"); mg_plan_destroy(p); return rc; }
        p->d_lit = d + 64;
    }
    if (rec_phase) TRY(upload(p, &p->d_rec_phase, rec_phase, n_rec, st));
    p->n_cseg = n_cseg;
    if (any_long) {
        TRY(upload(p, &p->d_crec_seg_off, c_rec_seg_off, n_rec + 1, st));
        TRY(upload(p, &p->d_cseg_contig, c_contig, n_cseg, st));
        TRY(upload(p, &p->d_cseg_start, c_start, n_cseg, st));
        TRY(upload(p, &p->d_cseg_end, c_end, n_cseg, st));
        TRY(upload(p, &p->d_cseg_strand, c_strand, n_cseg, st));
    } else {
        p->d_crec_seg_off = p->d_rec_seg_off; p->d_cseg_contig = p->d_seg_contig; p->d_cseg_start = p->d_seg_start;
        p->d_cseg_end = p->d_seg_end; p->d_cseg_strand = p->d_seg_strand;
    }
    p->stop_mask = MG_STD_STOPS;
    TRY(dalloc(p, &p->d_blk_r0, (p->n_piece + PLAN_TILE - 1) / PLAN_TILE + 1, st));
    {   // the nucleotide text size, from the clamped lengths above
        const int64_t up = nuc_bytes;
        p->nuc_upper = up;
        p->blk1k_cap = (up >> 10) + 3;
        TRY(dalloc(p, &p->d_blk1k, p->blk1k_cap, st));
    }
    TRY(dalloc(p, &p->d_piece_src, p->n_piece, st));
    TRY(dalloc(p, &p->d_piece_off, p->n_piece + 1, st));
    TRY(dalloc(p, &p->d_prot_off, n_rec + 1, st));
    TRY(dalloc(p, &p->d_rec_aa, n_rec, st));
    TRY(dalloc(p, &p->d_rec_skip, n_rec, st));
    // look-back scratch: [ticket, status per PLAN_TILE-piece block] [ticket, status per REC_TILE-record block] [nuc total, prot total];
    // the one-launch K1 uses two [ticket, status per PR_RECS-record block] arrays and the last two words
    p->scan_tmp_cap = (p->n_piece + PLAN_TILE - 1) / PLAN_TILE + 1 + 2 * ((n_rec + 127) / 128 + 1) + 2;
    for (int64_t r = 0; r < n_rec; r++) p->max_seg_per_rec = std::max(p->max_seg_per_rec, rec_seg_off[r + 1] - rec_seg_off[r]);
    TRY(dalloc(p, &p->d_scan_tmp, p->scan_tmp_cap, st));
#undef TRY
    if (n_rec > 0) {
        // record -> first piece block: a function of rec_seg_off alone, so it is computed here, once per table, and not in every
        // prepare (one launch less on the critical path of a step: ~4 us of a 74 us step at 8 GPUs)
        const int64_t n_block = (p->n_piece + PLAN_TILE - 1) / PLAN_TILE, n_rblock = (n_rec + 255) / 256;
        k_plan_block_rec<<<(unsigned)n_rblock, 256, 0, st>>>(n_block, n_rec, p->d_rec_seg_off, p->d_blk_r0);
        MG_COUNT_LAUNCH();
        if (cudaGetLastError() != cudaSuccess) { mg_set_error("k_plan_block_rec launch failed"); mg_plan_destroy(p); return MG_ECUDA; }
    }
    *out = p;
    return MG_OK;
}

extern "C" int mg_plan_destroy(mg_plan *p) {
    if (!p) return MG_OK;
    cudaSetDevice(p->device);
    mg_var_free(p);
    for (void *d : p->owned) cudaFreeAsync(d, p->last_stream);
    if (p->d_out) cudaFreeAsync(p->d_out, p->last_stream);
    delete p;
    return MG_OK;
}

// The plan's protein emits read their own translation table from here on.  It is built and uploaded now, so an emit queued or
// captured in a graph later reads a table that is already on the device; codon64 == NULL goes back to the genome's table.
extern "C" int mg_plan_set_codon_table(mg_plan *p, const uint8_t *codon64) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    if (!codon64) { p->own_code = false; p->stop_mask = MG_STD_STOPS; return MG_OK; }
    // the record pass drops a leading codon for trimX when it holds a base outside ACGT, i.e. where the table gives 'X'
    for (int c = 0; c < 64; c++) MG_REQUIRE(codon64[c] != 'X', "codon64 maps an A/C/G/T codon to 'X'");
    uint64_t stops = 0;
    for (int c = 0; c < 64; c++) if (codon64[c] == '*') stops |= 1ull << c;
    MG_CUDA(cudaSetDevice(p->device));
    uint8_t t[8192];
    build_aa4096(t, codon64);
    for (uint32_t c = 0; c < 4096; c++) t[4096 + mg_aa_slot(c)] = t[c];
    cudaStream_t st = p->last_stream;                 // after the emits already queued with the previous table
    if (!p->d_aa8192) {
        int rc = dalloc(p, &p->d_aa8192, 8192, st);
        if (rc) return rc;
    }
    MG_CUDA(cudaMemcpyAsync(p->d_aa8192, t, 8192, cudaMemcpyHostToDevice, st));
    MG_CUDA(cudaStreamSynchronize(st));
    p->own_code = true;
    p->stop_mask = stops;
    return MG_OK;
}

// K1, first half: clamp + lengths + offsets of every piece and record; the two text sizes land in p->d_totals
static int plan_alloc_tiles(mg_plan *p, int64_t cap_nuc, int64_t cap_prot, cudaStream_t st);
static int64_t plan_tile_need(int64_t cap_nuc, int64_t cap_prot) {   // tile table entries for texts of up to these sizes
    return (cap_nuc + MG_NUC_TILE - 1) / MG_NUC_TILE + 1 + (cap_prot + MG_PROT_TILE - 1) / MG_PROT_TILE + 1;
}
static int64_t pr_tiles(const mg_plan *p) { return (p->n_rec + PR_RECS - 1) / PR_RECS; }   // blocks of k_plan_rec

// scatter_tiles: the tile tables are sized for the caller's capacities and filled by the plan kernels themselves
static int plan_launch_records(mg_plan *p, cudaStream_t st);
static int plan_launch_scans(mg_plan *p, int prot_flags, cudaStream_t st, bool scatter_tiles = false, int64_t cap_nuc = 0,
                             int64_t cap_prot = 0) {
    mg_genome *g = p->g;
    p->prot_flags = prot_flags;
    p->last_stream = st;
    p->prot_ready = false;
    const int64_t n_block = (p->n_piece + PLAN_TILE - 1) / PLAN_TILE, n_rblock = (p->n_rec + REC_TILE - 1) / REC_TILE;
    unsigned long long *tmp_a = reinterpret_cast<unsigned long long *>(p->d_scan_tmp), *tmp_b = tmp_a + n_block + 1;
    p->d_totals = reinterpret_cast<int64_t *>(tmp_b + n_rblock + 1);
    // Each pass zeroes ITS OWN look-back words, in its own stream, right before its kernel: the record pass of a deferred
    // prepare may still be running on another stream when the next piece pass of the same plan starts (a bench step that
    // re-prepares a plan does exactly that), and wiping its ticket counter / status words would leave its tiles waiting for
    // predecessors for ever.  The two text sizes are written unconditionally by the last tile of each pass.
    // The one-launch K1 zeroes its two look-back arrays and not the totals either: the previous step's K3 or products kernel
    // may still read them on another stream to bound its tiles.  Only with no record (no kernel writes the totals) is all of
    // the scratch zeroed.
    const bool one_launch = p->n_rec > 0 && p->max_seg_per_rec <= PR_MAXSEG && mg_k1_mode() == 1;
    if (p->n_rec == 0) MG_CUDA(cudaMemsetAsync(p->d_scan_tmp, 0, p->scan_tmp_cap * sizeof(int64_t), st));
    else if (one_launch) MG_CUDA(cudaMemsetAsync(p->d_scan_tmp, 0, 2 * (pr_tiles(p) + 1) * sizeof(unsigned long long), st));
    else MG_CUDA(cudaMemsetAsync(tmp_a, 0, (n_block + 1) * sizeof(unsigned long long), st));
    int64_t *tf_nuc = nullptr, *tf_prot = nullptr;
    if (scatter_tiles) {
        int rc = plan_alloc_tiles(p, cap_nuc, cap_prot, st);
        if (rc) return rc;
        tf_nuc = p->d_nuc_tile;
        tf_prot = p->d_prot_tile;
    }
    if (p->n_rec == 0) { p->prot_ready = true; return MG_OK; }
    if (one_launch) {                                  // K1 in one launch
        const int64_t n_tile = pr_tiles(p);
        unsigned long long *ta = reinterpret_cast<unsigned long long *>(p->d_scan_tmp), *tb = ta + n_tile + 1;
        p->d_totals = reinterpret_cast<int64_t *>(p->d_scan_tmp + p->scan_tmp_cap - 2);
        k_plan_rec<<<(unsigned)n_tile, PR_THREADS, 0, st>>>(
            p->n_rec, p->n_piece, p->d_rec_seg_off, p->d_seg_contig, p->d_seg_start, p->d_seg_end, p->d_seg_strand, p->d_rec_lit_off,
            p->d_rec_pre, p->d_rec_suf, p->d_rec_phase, prot_flags, g->d_contig_len, g->d_contig_base, g->n_contigs, 2 * g->total_bases,
            g->d_packed, ta, tb, p->d_piece_off, p->d_piece_src, p->d_prot_off, p->d_rec_aa, p->d_rec_skip, p->d_totals, tf_nuc,
            p->n_nuc_tile, tf_prot, p->n_prot_tile, p->d_blk1k, p->blk1k_cap);
        MG_LAUNCH_CHECK();
        p->prot_ready = true;
        p->blk1k_ready = true;
        return MG_OK;
    }
    // (d_blk_r0 was filled by mg_plan_create.)  The 1 KB block table is read by the streaming K2 variant only.
    const bool want_blk1k = mg_emit_mode() == 2;
    p->blk1k_ready = want_blk1k;
    k_plan_pieces<<<(unsigned)n_block, PLAN_THREADS, 0, st>>>(
        p->n_piece, p->n_rec, p->d_rec_seg_off, p->d_blk_r0, p->d_seg_contig, p->d_seg_start, p->d_seg_end, p->d_seg_strand,
        p->d_rec_lit_off, p->d_rec_pre, p->d_rec_suf, g->d_contig_len, g->d_contig_base, g->n_contigs, 2 * g->total_bases,
        tmp_a, p->d_piece_off, p->d_piece_src, p->d_totals, tf_nuc, p->n_nuc_tile, p->d_blk1k, want_blk1k ? p->blk1k_cap : 0);
    MG_LAUNCH_CHECK();
    p->rec_tmp = tmp_b;
    p->rec_tmp_words = n_rblock + 1;
    p->rec_tile = tf_prot;
    if (prot_flags & MG_PROT_DEFER) return MG_OK;     // the record pass comes later (mg_plan_prepare_prot_async), maybe on another stream
    return plan_launch_records(p, st);
}

// K1, record half: amino-acid counts, first-codon trims and the offsets in the protein text (needed by the protein kernels only)
static int plan_launch_records(mg_plan *p, cudaStream_t st) {
    mg_genome *g = p->g;
    const int64_t n_rblock = (p->n_rec + REC_TILE - 1) / REC_TILE;
    MG_CUDA(cudaMemsetAsync(p->rec_tmp, 0, p->rec_tmp_words * sizeof(unsigned long long), st));
    k_plan_records<<<(unsigned)n_rblock, REC_THREADS, 0, st>>>(
        p->n_rec, p->d_rec_seg_off, p->d_piece_off, p->d_piece_src, g->d_packed, p->d_rec_phase, p->prot_flags,
        p->d_rec_aa, p->d_rec_skip, p->rec_tmp, p->d_prot_off, p->d_totals + 1, p->rec_tile, p->n_prot_tile);
    MG_LAUNCH_CHECK();
    p->prot_ready = true;
    return MG_OK;
}

// Emits and the calls that report what K1 computed need a plan prepared on the genome as it is now: K1's record pass read the
// first codons to fix trimX skips, amino-acid counts and protein offsets, and the emit kernels read the bases again.
int mg_plan_check_prepared(const mg_plan *p) {
    if (!p->prepared) { mg_set_error("mg_plan_prepare has not been called"); return MG_ESTATE; }
    if (p->generation != p->g->generation) {
        mg_set_error("the genome changed (pack, finalize or mask) since the plan was prepared: prepare it again");
        return MG_ESTATE;
    }
    return MG_OK;
}

// The record pass of a deferred prepare belongs to that prepare: after a genome change it fails like an emit (with the
// one-launch K1 the record pass has already run inside mg_plan_prepare_async).
extern "C" int mg_plan_prepare_prot_async(mg_plan *p, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    if (!p->prepared) { mg_set_error("mg_plan_prepare_async has not been called"); return MG_ESTATE; }
    if (const int rc0 = mg_plan_check_prepared(p)) return rc0;
    if (p->prot_ready || p->n_rec == 0) return MG_OK;
    MG_CUDA(cudaSetDevice(p->device));
    p->last_stream = (cudaStream_t)stream;
    if (p->totals_known) {                             // mg_plan_totals ran before this pass: its protein size (0) is stale
        p->prot_total = p->prot_cap;
        p->totals_known = false;
    }
    return plan_launch_records(p, (cudaStream_t)stream);
}

// K1, second half: tile -> first piece / first record, for texts of up to cap_nuc / cap_prot bytes (the real tile counts are
// derived on the device from p->d_totals).  Removes every global binary search from the emit kernels.
static int plan_alloc_tiles(mg_plan *p, int64_t cap_nuc, int64_t cap_prot, cudaStream_t st) {
    p->n_nuc_tile = (cap_nuc + MG_NUC_TILE - 1) / MG_NUC_TILE;
    p->n_prot_tile = (cap_prot + MG_PROT_TILE - 1) / MG_PROT_TILE;
    const int64_t tile_need = plan_tile_need(cap_nuc, cap_prot);
    if (tile_need > p->tile_cap) {                   // re-used when the same plan is prepared again
        void *d = nullptr;
        MG_CUDA(cudaMallocAsync(&d, tile_need * sizeof(int64_t), st));
        p->owned.push_back(d);
        p->d_tile_buf = (int64_t *)d;
        p->tile_cap = tile_need;
    }
    p->d_nuc_tile = p->d_tile_buf;
    p->d_prot_tile = p->d_tile_buf + p->n_nuc_tile + 1;
    return MG_OK;
}

static int plan_launch_tiles(mg_plan *p, int64_t cap_nuc, int64_t cap_prot, cudaStream_t st) {
    int rc = plan_alloc_tiles(p, cap_nuc, cap_prot, st);
    if (rc) return rc;
    if (p->n_rec > 0 && p->n_nuc_tile + p->n_prot_tile > 0) {
        k_plan_tiles<<<(unsigned)((p->n_nuc_tile + p->n_prot_tile + 2 + 255) / 256), 256, 0, st>>>(
            p->d_totals, p->d_piece_off, p->n_piece, MG_NUC_TILE, p->n_nuc_tile, p->d_nuc_tile, p->d_prot_off, p->n_rec, MG_PROT_TILE,
            p->n_prot_tile, p->d_prot_tile);
        MG_LAUNCH_CHECK();
    }
    return MG_OK;
}

static int plan_read_totals(mg_plan *p, cudaStream_t st, int64_t totals[2]) {
    totals[0] = totals[1] = 0;
    if (p->n_rec > 0) {
        MG_CUDA(cudaMemcpyAsync(totals, p->d_totals, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        MG_CUDA(cudaStreamSynchronize(st));
    }
    return MG_OK;
}

extern "C" int mg_plan_prepare(mg_plan *p, int prot_flags, int64_t *nuc_total, int64_t *prot_total, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    p->prepared = false;
    p->prepares++;
    int rc = plan_launch_scans(p, prot_flags & ~MG_PROT_DEFER, st);
    if (rc) return rc;
    int64_t totals[2];
    rc = plan_read_totals(p, st, totals);            // the one host round trip: the caller sizes its buffers from these
    if (rc) return rc;
    p->nuc_total = totals[0];
    p->prot_total = totals[1];
    p->totals_known = true;
    rc = plan_launch_tiles(p, p->nuc_total, p->prot_total, st);
    if (rc) return rc;
    p->prepared = true;
    p->generation = p->g->generation;
    if (nuc_total) *nuc_total = p->nuc_total;
    if (prot_total) *prot_total = p->prot_total;
    return MG_OK;
}

extern "C" int mg_plan_prepare_async(mg_plan *p, int prot_flags, int64_t nuc_capacity, int64_t prot_capacity, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    MG_REQUIRE(nuc_capacity >= 0 && prot_capacity >= 0, "capacities must be >= 0");
    MG_CUDA(cudaSetDevice(p->device));
    if (plan_tile_need(nuc_capacity, prot_capacity) > p->tile_cap) {
        const int rc0 = mg_refuse_growth_in_capture((cudaStream_t)stream, "mg_plan_prepare_async (first prepare, or larger capacities)");
        if (rc0) return rc0;
    }
    p->prepared = false;
    p->prepares++;
    int rc = plan_launch_scans(p, prot_flags, (cudaStream_t)stream, true, nuc_capacity, prot_capacity);
    if (rc) return rc;
    p->nuc_total = nuc_capacity;                     // until mg_plan_totals: what the caller's buffers can take
    p->prot_total = prot_capacity;
    p->prot_cap = prot_capacity;
    p->totals_known = false;
    p->prepared = true;
    p->generation = p->g->generation;
    return MG_OK;
}

extern "C" int mg_plan_totals(mg_plan *p, int64_t *nuc_total, int64_t *prot_total, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    if (const int rc0 = mg_plan_check_prepared(p)) return rc0;
    MG_CUDA(cudaSetDevice(p->device));
    if (!p->totals_known) {
        int64_t totals[2];
        int rc = plan_read_totals(p, (cudaStream_t)stream, totals);
        if (rc) return rc;
        if (!p->prot_ready) totals[1] = 0;               // deferred record pass not run: no protein text (the device word is stale)
        if (totals[0] > p->nuc_total || totals[1] > p->prot_total) {
            mg_set_error("text sizes (%lld nucleotide, %lld protein bytes) exceed the capacities given to mg_plan_prepare_async "
                         "(%lld, %lld): the emitted texts are truncated", (long long)totals[0], (long long)totals[1],
                         (long long)p->nuc_total, (long long)p->prot_total);
            return MG_EINVAL;
        }
        p->nuc_total = totals[0];
        p->prot_total = totals[1];
        p->totals_known = true;
        // the tile tables stay sized for the capacities: n_nuc_tile / n_prot_tile remain upper bounds of the grids
    }
    if (nuc_total) *nuc_total = p->nuc_total;
    if (prot_total) *prot_total = p->prot_total;
    return MG_OK;
}

extern "C" int mg_plan_lengths(mg_plan *p, int64_t *nuc_len, int64_t *aa_len, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    if (const int rc0 = mg_plan_check_prepared(p)) return rc0;
    if (p->n_rec == 0 || (!nuc_len && !aa_len)) return MG_OK;
    if (aa_len && !p->prot_ready) { mg_set_error("the record pass was deferred (MG_PROT_DEFER): call mg_plan_prepare_prot_async first"); return MG_ESTATE; }
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    int64_t *d = nullptr;
    MG_CUDA(cudaMallocAsync((void **)&d, 2 * p->n_rec * sizeof(int64_t), st));
    k_plan_lengths<<<(unsigned)((p->n_rec + 255) / 256), 256, 0, st>>>(p->n_rec, p->d_rec_seg_off, p->d_piece_off, p->d_rec_aa,
                                                                        d, d + p->n_rec);
    MG_LAUNCH_CHECK();
    if (nuc_len) MG_CUDA(cudaMemcpyAsync(nuc_len, d, p->n_rec * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    if (aa_len) MG_CUDA(cudaMemcpyAsync(aa_len, d + p->n_rec, p->n_rec * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MG_CUDA(cudaStreamSynchronize(st));
    MG_CUDA(cudaFreeAsync(d, st));
    return MG_OK;
}
