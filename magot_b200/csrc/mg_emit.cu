// mg_emit.cu -- K2 (segmented interval gather + per-segment reverse complement + FASTA framing) and
// K3 (codon translation of the spliced sequence).  Both are flat passes over OUTPUT bytes: one lane owns
// one aligned chunk of the final text (32 bytes in K2, 16 in K3) and issues exactly one vector store,
// so stores are perfectly coalesced and the load balance is independent of transcript/exon lengths.
//
//   K2 replaces ParentAnnotation.get_fasta seq_type="nucleotide" (genome.py:687-710),
//      BaseAnnotation.get_seq (genome.py:603-608) and Sequence.reverse_compliment (genome.py:784-793).
//   K3 replaces Sequence.translate(frame=0, strand='+', trimX=True) (genome.py:795-822) as called on
//      the spliced sequence at genome.py:707.
//
// Algorithmic HBM bytes (SURVEY 8d): K2 = 0.5 B/base packed read + 1 B/base text written (+ tables);
// K3 = 0.5 B/base read + 1/3 B/base written.  No dense contraction exists -> no tensor cores.
//
// How the kernels got here (ncu evidence under profiles/, A/B numbers in DESIGN.md section 5):
//   r1a  16 bytes/lane, per-chunk binary search, reverse complement in registers: issue-bound, 17 of 32 lanes active.
//   r1c  the genome keeps a second, reverse-complemented plane, so a '-' interval is a plain forward read (mg_common.cuh);
//        tile-relative tables in shared memory; the first two GENOME pieces of a chunk are handled branch-free.
//   r1j  32 bytes/lane with 256-bit stores, 32 KB tiles.
//   r1u  loads with .L2::64B (L2 otherwise fills whole 128-byte lines for ~96-byte pieces), staging cut to ~14 KB so that
//        8 CTAs are resident and most of the SM's 256 KB stays L1, FASTA framing written by the same CTA after a barrier
//        (no lane ever branches on framing, no second kernel), text sizes read from the device (mg_plan_prepare_async).
//   K3   the 48-nibble codon window is filled by a loop over the record's pieces (one one-sided mask each); the codon
//        table sits in shared memory in an order that makes a lookup one wavefront (mg_aa_slot).
#include <algorithm>
#include <cstring>
#include "mg_common.cuh"
#include "mg_gather.cuh"
#include "mg_emit_common.cuh"

#ifndef NUC_THREADS
#define NUC_THREADS 256
#endif
#ifndef NUC_LD64
#define NUC_LD64 1
#endif
#ifndef FRAME_BATCH
#define FRAME_BATCH 1
#endif
#ifndef FRAME_LANES4
#define FRAME_LANES4 1
#endif
#ifndef NUC_RC_COST
#define NUC_RC_COST 0
#endif
#ifndef NUC_FASTDEC
#define NUC_FASTDEC 1                                    // ACGT/acgt-only chunks take a two-look-up decode (mg_decode32)
#endif
#ifndef NUC_MINB
#define NUC_MINB 8                                       // 32 registers, 64 resident warps per SM
#endif
#ifndef NUC_CAP
#define NUC_CAP 768                                      // pieces staged per tile (a 32 KB tile of config 4 has ~200); small, so
                                                         // that 8 CTAs fit and most of the SM's 256 KB stays L1 cache (measured +7 %)
#endif
#define NUC_UNITS (MG_NUC_TILE / 32)
#define NUC_LITCAP 256                                   // literal pieces listed per tile (config 4: ~50)
#define NUC_CHUNKS ((MG_NUC_TILE / 32 + NUC_THREADS - 1) / NUC_THREADS)   // 4 chunks of 32 B per thread

#ifndef PROT_WIDE_SLOT
#define PROT_WIDE_SLOT 1
#endif
#ifndef PROT_THREADS
#define PROT_THREADS 256
#endif
#define PROT_CHUNKS (MG_PROT_TILE / 16 / PROT_THREADS)  // 4
#ifndef PROT_MINB
#define PROT_MINB 7                                      // 36 registers; measured 5: 0.147, 6: 0.136, 7: 0.129, 8: 0.130 ms
#endif
#ifndef PROT_RCAP
#define PROT_RCAP 256                                    // records staged per tile (a 16 KB tile of config 4 has ~45)
#endif
#ifndef PROT_PCAP
#define PROT_PCAP 768                                    // pieces staged per tile (~300); small for the same reason as NUC_CAP
#endif
#define PROT_UNITS (MG_PROT_TILE / 64)


// Slow path of K2, one 32-byte chunk assembled from EVERY staged piece that reaches into it, genome and literal alike:
// chunks that contain framing bytes (">ID\n", "\n"; ~1.5 per record), three or more pieces, or a byte outside the
// packed alphabet.  Takes scalars only, so the fast path keeps its words in registers.
__device__ __noinline__ void nuc_chunk_slow(const uint32_t *__restrict__ packed, const int64_t *s_base, const int32_t *s_rel,
                                            const uint8_t *s_kind, const uint16_t *s_unit, int ncache, int p, int end, int64_t T,
                                            const uint8_t *__restrict__ lit, const int64_t *__restrict__ exc_pos,
                                            const uint8_t *__restrict__ exc_byte, int64_t n_exc, uint8_t *__restrict__ dst) {
    uint32_t w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int k = s_unit[p >> 5];
    for (; k < ncache && s_rel[k] - p < end; k++) {
        const int lo = max(s_rel[k] - p, 0), hi = min(s_rel[k + 1] - p, end);
        if (hi <= lo) continue;
        const uint32_t m = (hi >= 32 ? 0xFFFFFFFFu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
        uint32_t b[8];
        if (s_kind[k] == 2) {
            ld_lit16(lit, s_base[k] + p, b);
            ld_lit16(lit, s_base[k] + p + 16, b + 4);
        } else {
            uint32_t n[4];
            const int64_t g = s_base[k] + p;
            ld_nib32(packed, g, n);
#pragma unroll
            for (int q = 0; q < 4; q++) mg_decode8(n[q], b[2 * q], b[2 * q + 1]);
            if (n_exc > 0 && g < T) {
                for (int q = lo; q < hi; q++) {
                    if (((n[q >> 3] >> ((q & 7) * 4)) & 15u) == MG_CODE_EXC) {
                        const uint32_t c = mg_exc_byte(exc_pos, exc_byte, n_exc, g + q);
                        b[q >> 2] = (b[q >> 2] & ~(0xFFu << ((q & 3) * 8))) | (c << ((q & 3) * 8));
                    }
                }
            }
        }
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const uint32_t mk = expand4(m >> (4 * q));
            w[q] = (w[q] & ~mk) | (b[q] & mk);
        }
    }
    st32_2x16(dst, w);
}

// ---- K2 ---------------------------------------------------------------------------------------------------------
// One lane = 32 output bytes = one 256-bit store.
//  * a chunk normally lies inside a run of genome pieces: X is the first genome piece that reaches into it, Y (if X ends
//    inside the chunk) the next one; both are fetched branch-free and merged with one boundary mask.  Framing bytes
//    (">ID\n", "\n") before, between or after them get whatever nibbles happen to be there: no lane ever branches on
//    "is there framing in my chunk" (doing so costs a ~300-instruction divergent path in almost every warp-iteration).
//  * after the tile's chunks are stored, the CTA writes the framing bytes of its tile over those positions, one thread
//    per literal piece.  The lines are still in L2, so this costs no DRAM traffic; as a separate kernel after K2 it was
//    0.028 ms per launch of config 4, assembling the framing chunks in a slow path inside K2 +17 % instructions.
// arguments of one nucleotide product (one plan); the text size lives on the device (written by K1): the grid may be larger
// than the text (mg_plan_prepare_async); cap = what the caller's buffer holds
struct NucArgs {
    const uint32_t *packed;
    const int64_t *piece_off, *piece_src;
    int64_t n_piece;
    const int64_t *tile_first, *total_dev;
    int64_t cap, T;
    const uint8_t *lit;
    const int64_t *exc_pos;
    const uint8_t *exc_byte;
    int64_t n_exc;
    uint8_t *out;
};
// pieces of the tile: piece i covers text [s_rel[i], s_rel[i+1]) relative to the tile; the nibble index (literal: byte
// index) of tile position q is s_base[i] + q; s_ng[i] = first non-empty GENOME piece at or after i
template <int CAP>
struct NucSmemT {
    int64_t s_base[CAP + 2];
    int32_t s_rel[CAP + 3];
    uint16_t s_ng[CAP + 2];
    uint8_t s_kind[CAP + 2];
    uint16_t s_unit[NUC_UNITS];                       // piece holding byte 32*u of the tile, i.e. the first byte of chunk u
    uint16_t s_lits[NUC_LITCAP];                      // the tile's non-empty literal pieces (any order)
    int s_nlit;
};
typedef NucSmemT<NUC_CAP> NucSmem;

// one CTA, one 32 KB tile of the nucleotide text (the caller has checked tile * MG_NUC_TILE < total).  STAGE: the merged
// nibbles of every chunk are also left in shared memory (s_nib[8 + 4 * chunk ..], the K23 protein phase reads its codons there);
// *s_over is set when a chunk of the tile went through the generic path (its nibbles are then not staged).
template <bool STAGE, int CAP>
__device__ __forceinline__ void nuc_tile(const NucArgs &a, NucSmemT<CAP> &sm, const int64_t tile, const int64_t total, uint32_t *s_nib = nullptr,
                                         int *s_over = nullptr) {
    const uint32_t *__restrict__ packed = a.packed;
    const int64_t *__restrict__ piece_off = a.piece_off, *__restrict__ piece_src = a.piece_src;
    const int64_t n_piece = a.n_piece, T = a.T, n_exc = a.n_exc;
    const int64_t *__restrict__ tile_first = a.tile_first;
    const uint8_t *__restrict__ lit = a.lit;
    const int64_t *__restrict__ exc_pos = a.exc_pos;
    const uint8_t *__restrict__ exc_byte = a.exc_byte;
    uint8_t *__restrict__ out = a.out;
    int64_t *s_base = sm.s_base;
    int32_t *s_rel = sm.s_rel;
    uint16_t *s_ng = sm.s_ng, *s_unit = sm.s_unit, *s_lits = sm.s_lits;
    uint8_t *s_kind = sm.s_kind;
    int &s_nlit = sm.s_nlit;
    const int64_t P0 = tile * MG_NUC_TILE;
    const int64_t p_lo = tile_first[tile];
    int64_t p_hi = tile_first[tile + 1] + 1;          // one past the last piece this tile can touch
    if (p_hi > n_piece) p_hi = n_piece;
    const int ncache = (int)min((int64_t)CAP, p_hi - p_lo);
    const int tile_len = (int)min((int64_t)MG_NUC_TILE, total - P0);
    if (threadIdx.x == 0) s_nlit = 0;
    for (int i = threadIdx.x; i < ncache + 2; i += NUC_THREADS) {
        if (i < ncache) {
            const int64_t rel = __ldg(piece_off + p_lo + i) - P0;      // > -2^31: piece lengths are int32
            const int64_t nxt = __ldg(piece_off + p_lo + i + 1) - P0;
            const uint64_t sk = (uint64_t)__ldg(piece_src + p_lo + i);
            s_rel[i] = rel > MG_NUC_TILE ? MG_NUC_TILE : (int32_t)rel;
            s_base[i] = (int64_t)(sk & MG_SRC_MASK) - rel;
            s_kind[i] = nxt == rel ? PIECE_E : ((sk >> MG_KIND_SHIFT) == MG_KIND_LIT ? PIECE_L : PIECE_G);
        } else {
            const int64_t rel = i == ncache ? __ldg(piece_off + p_lo + ncache) - P0 : (int64_t)BIG;
            s_rel[i] = rel > MG_NUC_TILE ? (i == ncache ? MG_NUC_TILE : BIG) : (int32_t)rel;
            s_base[i] = 0;
            s_kind[i] = PIECE_G;
        }
    }
    if (threadIdx.x == 0) s_rel[ncache + 2] = BIG;
    __syncthreads();
    for (int i = threadIdx.x; i < ncache + 2; i += NUC_THREADS) {
        int k = i;
        while (k < ncache && s_kind[k] != PIECE_G) k++;               // runs of literal / empty pieces are short
        s_ng[i] = (uint16_t)k;
        if (i < ncache) {
            const int r0 = s_rel[i] < 0 ? 0 : s_rel[i], r1 = s_rel[i + 1] < 0 ? 0 : s_rel[i + 1];
            const int u1 = min((r1 + 31) >> 5, NUC_UNITS);
            for (int u = (r0 + 31) >> 5; u < u1; u++) s_unit[u] = (uint16_t)i;
            if (s_kind[i] == PIECE_L && r1 > r0) {
                const int slot = atomicAdd(&s_nlit, 1);
                if (slot < NUC_LITCAP) s_lits[slot] = (uint16_t)i;
            }
        }
    }
    __syncthreads();
    const int covered = s_rel[ncache];                // tile-relative position where the staged pieces end

#pragma unroll 1
    for (int cidx = 0; cidx < NUC_CHUNKS; cidx++) {
        const int p = (cidx * NUC_THREADS + (int)threadIdx.x) << 5;
        if (p >= tile_len) break;
        if (p + 32 > covered && covered < tile_len) {  // staging overflowed: slow path straight from global memory
            const int64_t j = mg_search_le(piece_off, p_lo, n_piece, P0 + p);
            nuc_chunk_generic(packed, piece_off, piece_src, j, P0 + p, total, T, lit, exc_pos, exc_byte, n_exc, out);
            if (STAGE) *s_over = 1;
            continue;
        }
        const int A = s_unit[p >> 5];                  // the (non-empty) piece that holds byte p
        const int end = min(32, tile_len - p);
        const int X = s_ng[A];
        const bool hasX = s_rel[X] - p < end;
        const int hiX = s_rel[X + 1] - p;              // X covers chunk positions [.., hiX)
        const int Y = s_ng[X + 1];
        const bool hasY = hasX && hiX < end && s_rel[Y] - p < end;
        const bool more = hasY && s_rel[Y + 1] - p < end;              // Y ends inside the chunk: a third genome piece may follow
        uint32_t rare = 0;
        const int64_t gx = hasX ? s_base[X] + p : (int64_t)MG_FRONT_PAD;
        const int64_t gy = hasY ? s_base[Y] + p : (int64_t)MG_FRONT_PAD;
        const uint32_t *qx = packed + (gx >> 3), *qy = packed + (gy >> 3);
        uint32_t rx[5], ry[5];
        ld_pk5(qx, rx);
        ld_pk5(qy, ry);
        const uint32_t shx = ((uint32_t)gx & 7u) << 2, shy = ((uint32_t)gy & 7u) << 2;
        const int c = hiX > 32 ? 32 : hiX;
        uint32_t n[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {                  // positions < hiX come from X, the rest from Y
            const int t = c - 8 * k;
            const uint32_t m = low_nibbles(t);
            n[k] = (__funnelshift_r(rx[k], rx[k + 1], shx) & m) | (__funnelshift_r(ry[k], ry[k + 1], shy) & ~m);
        }
        // Further genome pieces inside the same 32 bytes (a segment of a few bases: 0.1-0.2 % of the chunks of config 4, but
        // some lane of 3-7 % of the warps): each one overwrites the chunk from its first position on, as in K3.  This used to
        // go through the generic per-piece path (~7 % of the kernel's instructions).
        if (more) {
#pragma unroll 1
            for (int Z = s_ng[Y + 1]; s_rel[Z] - p < end; Z = s_ng[Z + 1]) {
                const int cz = s_rel[Z] - p;                           // > 0: Z starts after Y inside the chunk
                const int64_t gz = s_base[Z] + p;
                const uint32_t *qz = packed + (gz >> 3);
                const uint32_t shz = ((uint32_t)gz & 7u) << 2;
                uint32_t rz[5];
                ld_pk5(qz, rz);
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const uint32_t keep = low_nibbles(cz - 8 * k);
                    n[k] = (n[k] & keep) | (__funnelshift_r(rz[k], rz[k + 1], shz) & ~keep);
                }
            }
        }
        // code 15 = byte outside the packed alphabet on a '+' piece (the reverse plane already holds 'n',
        // genome.py:791-792): the exact byte the FASTA had must come out (genome.py:606 keeps it).  Rare.
        if (n_exc > 0) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t e = n[k] & (n[k] >> 1);
                rare |= e & (e >> 2) & 0x11111111u;
            }
        }
        if (STAGE) *reinterpret_cast<uint4 *>(s_nib + 8 + (p >> 3)) = make_uint4(n[0], n[1], n[2], n[3]);
        if (rare) {
            nuc_chunk_slow(packed, s_base, s_rel, s_kind, s_unit, ncache, p, end, T, lit, exc_pos, exc_byte, n_exc, out + P0 + p);
            continue;
        }
#if NUC_RC_COST
        // A/B knob (profiles/README.md, "reverse-complement plane"): the ALU work a register reverse complement of this chunk
        // would cost, applied twice (identity) to EVERY chunk, i.e. about twice what a 50 % '-' strand mix would pay without
        // the second plane -- the memory side (a descending window instead of an ascending one) is the same traffic
        {
            const uint64_t a = mg_rc_nib16(mg_rc_nib16(((uint64_t)n[1] << 32) | n[0]));
            const uint64_t b = mg_rc_nib16(mg_rc_nib16(((uint64_t)n[3] << 32) | n[2]));
            n[0] = (uint32_t)a; n[1] = (uint32_t)(a >> 32); n[2] = (uint32_t)b; n[3] = (uint32_t)(b >> 32);
        }
#endif
        uint32_t w[8];
#if NUC_FASTDEC
        mg_decode32(n, w);
#else
#pragma unroll
        for (int k = 0; k < 4; k++) mg_decode8(n[k], w[2 * k], w[2 * k + 1]);
#endif
        st32(out + P0 + p, w);
    }

    // framing bytes of this tile, over the placeholders the chunks above left (same CTA, ordered by the barrier): eight lanes
    // per literal piece, so the ~50 pieces of a tile are written by all warps at once
    __syncthreads();
    const int nlit = s_nlit;
    if (nlit <= NUC_LITCAP) {
        for (int k = threadIdx.x; k < nlit * 8; k += NUC_THREADS) {
            const int i = s_lits[k >> 3];
            const int r1 = min(s_rel[i + 1], tile_len);
            const uint8_t *src = lit + s_base[i];
#if FRAME_BATCH
            // four loads in flight per lane before the first store (a header of <= 32 bytes is ONE load latency, not three,
            // at the very end of the CTA's life)
            for (int q = max(s_rel[i], 0) + (k & 7); q < r1; q += 32) {
                uint8_t b[4];
#pragma unroll
                for (int j = 0; j < 4; j++) b[j] = q + 8 * j < r1 ? __ldg(src + q + 8 * j) : (uint8_t)0;
#pragma unroll
                for (int j = 0; j < 4; j++) if (q + 8 * j < r1) out[P0 + q + 8 * j] = b[j];
            }
#else
            for (int q = max(s_rel[i], 0) + (k & 7); q < r1; q += 8) out[P0 + q] = __ldg(src + q);
#endif
        }
    } else {                                          // more literal pieces than the list holds: one thread per piece
        for (int i = threadIdx.x; i < ncache; i += NUC_THREADS) {
            if (s_kind[i] != PIECE_L) continue;
            const int r0 = max(s_rel[i], 0), r1 = min(s_rel[i + 1], tile_len);
            const uint8_t *src = lit + s_base[i];
            for (int q = r0; q < r1; q++) out[P0 + q] = __ldg(src + q);
        }
    }
}

__global__ void __launch_bounds__(NUC_THREADS, NUC_MINB) k_emit_nuc(const __grid_constant__ NucArgs a) {
    const int64_t total = min(__ldg(a.total_dev), a.cap);
    if ((int64_t)blockIdx.x * MG_NUC_TILE >= total) return;
    __shared__ NucSmem sm;
    nuc_tile<false, NUC_CAP>(a, sm, blockIdx.x, total);
}


// Output chunk = 16 bytes of protein text.  Amino acid a of record r is the codon at spliced offset
// skip[r] + 3a; the 4096-entry nibble-triplet table (case-insensitive, anything non-ACGT -> 'X') sits in
// shared memory.  Stop codons are emitted as '*' and translation continues (genome.py:811-818).
struct ProtArgs {
    const uint32_t *packed;
    const int64_t *piece_off, *piece_src, *rec_seg_off, *prot_off;
    const int32_t *rec_aa;
    const int8_t *rec_skip;
    const int32_t *rec_pre, *rec_suf;
    const int64_t *rec_lit_off;
    const uint8_t *lit;
    int64_t n_rec;
    const int64_t *tile_first, *total_dev;
    int64_t cap;
    const uint8_t *aa4096, *aa4096h;
    uint8_t *out;
};
struct ProtSmem {
    __align__(16) uint8_t s_aa[4096];
    // records of the tile: residues occupy protein-text positions [r_s[i], r_e[i]) relative to the tile (empty when the
    // record has none); r_q0 = nucleotide-text position (relative to O) of the codon that would land on tile position 0;
    // r_j0 = first segment piece of the record (tile-local index)
    int32_t r_s[PROT_RCAP + 2], r_e[PROT_RCAP + 2], r_q0[PROT_RCAP + 2];
    int16_t r_j0[PROT_RCAP + 2];
    // pieces of those records: piece i covers nucleotide-text [s_rel[i], s_rel[i+1]) relative to O
    int64_t s_base[PROT_PCAP + 4];
    int32_t s_rel[PROT_PCAP + 5];
    uint16_t s_unit[PROT_UNITS];
};

// one CTA, one 16 KB tile of the protein text (the caller has checked tile * MG_PROT_TILE < total)
__device__ __forceinline__ void prot_tile(const ProtArgs &a, ProtSmem &sm, const int64_t tile, const int64_t total) {
    const uint32_t *__restrict__ packed = a.packed;
    const int64_t *__restrict__ piece_off = a.piece_off, *__restrict__ piece_src = a.piece_src;
    const int64_t *__restrict__ rec_seg_off = a.rec_seg_off, *__restrict__ prot_off = a.prot_off;
    const int32_t *__restrict__ rec_aa = a.rec_aa;
    const int8_t *__restrict__ rec_skip = a.rec_skip;
    const int32_t *__restrict__ rec_pre = a.rec_pre, *__restrict__ rec_suf = a.rec_suf;
    const int64_t *__restrict__ rec_lit_off = a.rec_lit_off;
    const uint8_t *__restrict__ lit = a.lit;
    const int64_t n_rec = a.n_rec;
    const int64_t *__restrict__ tile_first = a.tile_first;
    const uint8_t *__restrict__ aa4096 = a.aa4096, *__restrict__ aa4096h = a.aa4096h;
    uint8_t *__restrict__ out = a.out;
    uint8_t *s_aa = sm.s_aa;
    int32_t *r_s = sm.r_s, *r_e = sm.r_e, *r_q0 = sm.r_q0, *s_rel = sm.s_rel;
    int16_t *r_j0 = sm.r_j0;
    int64_t *s_base = sm.s_base;
    uint16_t *s_unit = sm.s_unit;
    reinterpret_cast<uint4 *>(s_aa)[threadIdx.x] = __ldg(reinterpret_cast<const uint4 *>(aa4096h) + threadIdx.x);   // mg_aa_slot order
    const int64_t P0 = tile * MG_PROT_TILE;
    const int64_t r_lo = tile_first[tile];
    int64_t r_hi = tile_first[tile + 1] + 1;
    if (r_hi > n_rec) r_hi = n_rec;
    const int nrec = (int)(r_hi - r_lo);
    const int64_t pc_lo = __ldg(rec_seg_off + r_lo) + 2 * r_lo;
    const int64_t pc_hi = __ldg(rec_seg_off + r_hi) + 2 * r_hi;
    const int64_t O = __ldg(piece_off + pc_lo);
    const int64_t nraw64 = pc_hi - pc_lo;
    const bool fits = nrec <= PROT_RCAP && nraw64 <= PROT_PCAP && (__ldg(piece_off + pc_hi) - O) < (int64_t)BIG;
    const int tile_len = (int)min((int64_t)MG_PROT_TILE, total - P0);
    if (!fits) {                                      // rare: whole tile through the generic path
        for (int cidx = 0; cidx < PROT_CHUNKS; cidx++) {
            const int p = (cidx * PROT_THREADS + (int)threadIdx.x) << 4;
            if (p >= tile_len) break;
            const int64_t r = mg_search_le(prot_off, r_lo, n_rec, P0 + p);
            prot_chunk_generic(packed, piece_off, piece_src, rec_seg_off, prot_off, rec_aa, rec_skip, rec_pre, r, P0 + p, total,
                               aa4096, out);
        }
        __syncthreads();
        if (lit) prot_write_framing(r_lo, r_hi, P0, tile_len, prot_off, rec_aa, rec_lit_off, rec_pre, rec_suf, lit, out);
        return;
    }
    const int nraw = (int)nraw64;
    for (int i = threadIdx.x; i < nraw + 4; i += PROT_THREADS) {
        if (i <= nraw) {
            const int32_t rel = (int32_t)(__ldg(piece_off + pc_lo + i) - O);
            s_rel[i] = rel;
            s_base[i] = i < nraw ? (int64_t)((uint64_t)__ldg(piece_src + pc_lo + i) & MG_SRC_MASK) - rel : 0;
        } else {
            s_rel[i] = BIG;
            s_base[i] = 0;
        }
    }
    if (threadIdx.x == 0) s_rel[nraw + 4] = BIG;
    for (int i = threadIdx.x; i < nrec + 2; i += PROT_THREADS) {
        if (i < nrec) {
            const int64_t r = r_lo + i;
            int32_t naa = rec_aa[r];
            if (naa < 0) naa = 0;
            const int64_t rs = __ldg(prot_off + r) + rec_pre[r] - P0, re = rs + naa;
            const int64_t f0 = __ldg(rec_seg_off + r) + 2 * r;
            r_s[i] = rs < -BIG ? -BIG : (rs > MG_PROT_TILE ? MG_PROT_TILE : (int32_t)rs);
            r_e[i] = re < -BIG ? -BIG : (re > MG_PROT_TILE ? MG_PROT_TILE : (int32_t)re);
            r_q0[i] = (int32_t)(__ldg(piece_off + f0 + 1) - O) + rec_skip[r] - 3 * (int32_t)rs;
            r_j0[i] = (int16_t)(f0 + 1 - pc_lo);
        } else {
            r_s[i] = BIG; r_e[i] = BIG; r_q0[i] = 0; r_j0[i] = (int16_t)(nraw + 1);   // so that r_j0[R+1]-2 is the last record's suffix piece
        }
    }
    __syncthreads();
    // unit u -> first record whose residues end after byte 64*u
    for (int i = threadIdx.x; i <= nrec; i += PROT_THREADS) {
        int e0 = 0;
        if (i) { e0 = r_e[i - 1]; if (e0 < 0) e0 = 0; }
        int e1 = i < nrec ? r_e[i] : MG_PROT_TILE;
        if (e1 < 0) e1 = 0;
        const int u1 = min((e1 + 63) >> 6, PROT_UNITS);
        for (int u = i ? ((e0 + 63) >> 6) : 0; u < u1; u++) s_unit[u] = (uint16_t)i;
    }
    __syncthreads();

#pragma unroll 1
    for (int cidx = 0; cidx < PROT_CHUNKS; cidx++) {
        const int p = (cidx * PROT_THREADS + (int)threadIdx.x) << 4;
        if (p >= tile_len) break;
        int R = s_unit[p >> 6];
        while (r_e[R] <= p) R++;                      // first record whose residues end after byte p
        uint32_t bw[4] = {0, 0, 0, 0};
        // Usually ONE record has residues in the chunk: 16 codons = 48 spliced nibbles, taken from at most two
        // adjacent segment pieces and merged with one boundary mask, branch-free.  A second record in the same 16 bytes
        // needs >= 11 framing bytes in between, i.e. it happens for ~1 % of chunks, and takes another trip of the loop.
        for (; r_s[R] < p + 16; R++) {
            const int lo = max(r_s[R] - p, 0), hi = min(r_e[R] - p, 16);
            if (hi <= lo) continue;                   // record without residues
            // nucleotide-text position (relative to O) of the codon that lands on chunk position 0
            const int q = r_q0[R] + 3 * p;
            const int need_lo = q + 3 * lo, need_hi = q + 3 * hi;        // nibbles [need_lo, need_hi)
            int X;
            {   // last segment piece of the record that starts at or before need_lo (its pieces are adjacent)
                int a = r_j0[R], b = r_j0[R + 1] - 2; // b = one past the record's last segment piece
                while (b - a > 1) {
                    const int mid = (a + b) >> 1;
                    if (s_rel[mid] <= need_lo) a = mid; else b = mid;
                }
                X = a;
            }
            // The 48 nibbles come from the record's consecutive segment pieces, left to right: each piece overwrites the
            // window from its first nibble on (one one-sided mask), so one, two or more pieces are the same code.  One trip
            // for 73 % of the lanes of config 4, two for 26 %, more for the rest (a separate three-piece slow path was
            // entered by some lane in 43 % of the warp-iterations and cost 17 % of the kernel).
            uint32_t n[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll 1
            for (int j = X; s_rel[j] < need_hi; j++) {
                const int c = s_rel[j] - q;               // first window nibble this piece provides (<= 0 for the first piece)
                if (s_rel[j + 1] - q <= c) continue;      // empty piece
                const int64_t g = s_base[j] + q;
                const uint32_t *pp = packed + (g >> 3);
                const uint32_t sh = ((uint32_t)g & 7u) << 2;
                uint32_t v[7];
#pragma unroll
                for (int k = 0; k < 7; k++) v[k] = ld_pk(pp + k);
#pragma unroll
                for (int k = 0; k < 6; k++) {
                    const int t = c - 8 * k;
                    const uint32_t keep = low_nibbles(t);     // nibbles before the piece
                    n[k] = (n[k] & keep) | (__funnelshift_r(v[k], v[k + 1], sh) & ~keep);
                }
            }
            uint32_t w[4] = {0, 0, 0, 0};
#if PROT_WIDE_SLOT
            // mg_aa_slot for all 16 codons at once: slot = c ^ ((c >> 6) & 0xC) moves bits 8-9 of every 12-bit codon onto its
            // bits 2-3, i.e. the whole 192-bit window XORs itself shifted right by 6 under a mask with period 12
            {
                constexpr uint32_t M0 = 0x0C00C00Cu, M1 = 0xC00C00C0u, M2 = 0x00C00C00u;   // bits b with b % 12 in {2, 3}, words 0..2 (period 3 words)
                const uint32_t x0 = n[0] ^ (__funnelshift_r(n[0], n[1], 6) & M0), x1 = n[1] ^ (__funnelshift_r(n[1], n[2], 6) & M1),
                               x2 = n[2] ^ (__funnelshift_r(n[2], n[3], 6) & M2), x3 = n[3] ^ (__funnelshift_r(n[3], n[4], 6) & M0),
                               x4 = n[4] ^ (__funnelshift_r(n[4], n[5], 6) & M1), x5 = n[5] ^ ((n[5] >> 6) & M2);
                n[0] = x0; n[1] = x1; n[2] = x2; n[3] = x3; n[4] = x4; n[5] = x5;
            }
#pragma unroll
            for (int k = 0; k < 16; k++) {            // codon k = nibbles 3k..3k+2 = bits 12k.. of n[5]:..:n[0]
                const int bit = 12 * k, ww = bit >> 5, sh = bit & 31;
                const uint32_t idx = (sh > 20 ? __funnelshift_r(n[ww], n[ww + 1], sh) : (n[ww] >> sh)) & 0xFFFu;
                w[k >> 2] |= (uint32_t)s_aa[idx] << ((k & 3) * 8);
            }
#else
#pragma unroll
            for (int k = 0; k < 16; k++) {            // codon k = nibbles 3k..3k+2 = bits 12k.. of n[5]:..:n[0]
                const int bit = 12 * k, ww = bit >> 5, sh = bit & 31;
                uint32_t idx = n[ww] >> sh;
                if (sh > 20) idx |= n[ww + 1] << (32 - sh);
                w[k >> 2] |= (uint32_t)s_aa[mg_aa_slot(idx)] << ((k & 3) * 8);
            }
#endif
            const uint32_t m = ((1u << hi) - 1u) & ~((1u << lo) - 1u);
            if (m == 0xFFFFu) { bw[0] = w[0]; bw[1] = w[1]; bw[2] = w[2]; bw[3] = w[3]; }
            else {
#pragma unroll
                for (int k = 0; k < 4; k++) { const uint32_t mk = expand4(m >> (4 * k)); bw[k] = (bw[k] & ~mk) | (w[k] & mk); }
            }
        }
        mg_st16(out + P0 + p, bw[0], bw[1], bw[2], bw[3]);
    }
    __syncthreads();
    if (lit) prot_write_framing(r_lo, r_hi, P0, tile_len, prot_off, rec_aa, rec_lit_off, rec_pre, rec_suf, lit, out);
}

__global__ void __launch_bounds__(PROT_THREADS, PROT_MINB) k_emit_prot(const __grid_constant__ ProtArgs a) {
    const int64_t total = min(__ldg(a.total_dev), a.cap);   // on the device, see k_emit_nuc
    if ((int64_t)blockIdx.x * MG_PROT_TILE >= total) return;
    __shared__ ProtSmem sm;
    prot_tile(a, sm, blockIdx.x, total);
}


// ---- K23: spliced nucleotide text AND its translation in one pass ----------------------------------------------------------
// ParentAnnotation.get_fasta translates the very string it has just joined (genome.py:704-707): seq = "".join(child.get_seq())
// then Sequence(seq).translate().  K2 + K3 as two launches fetch the CDS bases from DRAM twice (config 4, ncu: 241 + 258 MB read)
// and K3 repeats the whole piece search / gather.  Here the CTA that assembles a 32 KB tile of the nucleotide text keeps the
// merged nibbles of the tile in shared memory (16 KB), and after the barrier that already precedes the framing bytes the same
// CTA translates every codon that STARTS in its tile from there:
//   * ownership: a protein byte belongs to the tile that holds its key position in the nucleotide text -- residue a of record r:
//     the first base of its codon; the ">ID\n" prefix: the first byte of the record's nucleotide text; the "\n" suffix: the first
//     byte of the nucleotide suffix.  Keys ascend along the protein text, so a tile owns one contiguous range [A, B) of it and
//     B(tile) = A(tile + 1): both ends are computed from the record that holds the tile's first byte (one warp each, a 32-ary
//     search of the record table while the other warps stage the pieces).
//   * a lane owns one aligned 16-byte chunk of that range (one st.v4 if the chunk lies inside [A, B); byte stores at the two
//     ends, which the neighbouring tiles share); its 16 codons are 48 nibbles at one offset of the staged tile: seven LDS and six
//     funnel shifts replace K3's search over the record's pieces and its 7-word global gather per piece.
//   * the one codon per tile that straddles the tile's end takes its last one or two bases from global memory (mg_gather_nib).
//   * tiles whose piece or record lists overflow the staging go through a per-residue global gather (always correct, slow).
#ifndef K23_RCAP
#define K23_RCAP 254                                  // records staged per tile (a 32 KB tile of config 4 holds ~30)
#endif
#ifndef K23_MINB
#define K23_MINB 6
#endif
#ifndef K23_CAP
#define K23_CAP NUC_CAP                              // pieces staged per tile in the fused kernel
#endif
#define K23_PMAX (MG_NUC_TILE / 3 + 64 * K23_RCAP + 64)   // the protein range of a tile that stays on the fast path (else per-residue path)
#define K23_NIBW (MG_NUC_TILE / 8 + 16)               // staged nibble words: the tile + 8 words of slack at both ends

struct FusedArgs {
    NucArgs n;
    ProtArgs p;
};
struct FusedSmem {
    union {
        NucSmemT<K23_CAP> n;                         // phase 1
        struct {                                     // phase 2
            __align__(16) uint8_t s_aa[4096];
            int32_t r_s[K23_RCAP + 2], r_e[K23_RCAP + 2], r_q0[K23_RCAP + 2];   // owned residues [r_s, r_e) relative to Abase; codon of position x at r_q0 + 3x
        } p;
    } u;
    __align__(16) uint32_t s_nib[K23_NIBW];
    int64_t s_bound[2][2];                           // [0]: R0, A   [1]: R1, B
    int s_over;
};

// record that owns piece `pc` (F(r) = rec_seg_off[r] + 2r <= pc < F(r+1)): 32-ary search by one warp
__device__ __forceinline__ int64_t k23_record_of_piece(const int64_t *__restrict__ rec_seg_off, int64_t n_rec, int64_t pc, int lane) {
    int64_t lo = 0, hi = n_rec;                      // answer in [lo, hi)
    while (hi - lo > 1) {
        const int64_t step = (hi - lo + 31) / 32;
        const int64_t r = lo + (int64_t)lane * step;
        const bool le = r < hi && __ldg(rec_seg_off + r) + 2 * r <= pc;
        const unsigned int b = __ballot_sync(0xffffffffu, le);        // lane 0 always true (F(lo) <= pc)
        const int k = 31 - __clz(b);
        lo = lo + (int64_t)k * step;
        hi = min(hi, lo + step);
    }
    return lo;
}

// protein bytes of record r whose key lies before nucleotide-text position Pb, plus prot_off[r]: the first protein byte that the
// tile starting at Pb owns
__device__ __forceinline__ int64_t k23_prot_pos(const ProtArgs &a, int64_t r, int64_t Pb) {
    const int64_t f0 = __ldg(a.rec_seg_off + r) + 2 * r, f1 = __ldg(a.rec_seg_off + r + 1) + 2 * (r + 1);
    const int64_t start = __ldg(a.piece_off + f0), ns = __ldg(a.piece_off + f0 + 1), sufpos = __ldg(a.piece_off + f1 - 1), end = __ldg(a.piece_off + f1);
    int64_t naa = a.rec_aa[r];
    if (naa < 0) naa = 0;
    const int64_t c0 = ns + a.rec_skip[r];
    int64_t before = Pb > c0 ? (Pb - c0 + 2) / 3 : 0;                  // codons that start before Pb
    if (before > naa) before = naa;
    return __ldg(a.prot_off + r) + (start < Pb ? ns - start : 0) + before + (sufpos < Pb ? end - sufpos : 0);
}

// one residue through the generic global gather (codon at nucleotide-text position S of record r)
__device__ __noinline__ uint8_t k23_residue_generic(const ProtArgs &a, int64_t r, int64_t S) {
    const int64_t f0 = __ldg(a.rec_seg_off + r) + 2 * r, f1 = __ldg(a.rec_seg_off + r + 1) + 2 * (r + 1);
    const int64_t j = mg_search_le(a.piece_off, f0 + 1, f1 - 1, S);
    uint64_t acc[3];
    mg_gather_nib(a.packed, a.piece_off, a.piece_src, j, S, 3, acc);
    return __ldg(a.aa4096 + ((uint32_t)acc[0] & 0xFFFu));
}

__global__ void __launch_bounds__(NUC_THREADS, K23_MINB) k_emit_nuc_prot(const __grid_constant__ FusedArgs f) {
    const int64_t total = min(__ldg(f.n.total_dev), f.n.cap);
    const int64_t tile = blockIdx.x;
    if (tile * MG_NUC_TILE >= total) return;
    __shared__ FusedSmem sm;
    const ProtArgs &a = f.p;
    const int64_t total_p = min(__ldg(a.total_dev), a.cap);
    const int64_t P0 = tile * MG_NUC_TILE;
    const int tile_len = (int)min((int64_t)MG_NUC_TILE, total - P0);
    const bool last_tile = P0 + MG_NUC_TILE >= total;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) sm.s_over = 0;
    // warps 0 / 1: record and first owned protein byte of this tile / of the next one (hidden behind the staging of the others)
    if (wid < 2 && !(wid == 1 && last_tile)) {
        const int64_t pc = __ldg(f.n.tile_first + tile + wid);
        const int64_t r = k23_record_of_piece(a.rec_seg_off, a.n_rec, pc, lane);
        if (lane == 0) {
            sm.s_bound[wid][0] = r;
            sm.s_bound[wid][1] = k23_prot_pos(a, r, P0 + (int64_t)wid * MG_NUC_TILE);
        }
    } else if (wid == 1 && lane == 0) {
        sm.s_bound[1][0] = a.n_rec - 1;
        sm.s_bound[1][1] = total_p;
    }
    nuc_tile<true, K23_CAP>(f.n, sm.u.n, tile, total, sm.s_nib, &sm.s_over);
    __syncthreads();                                  // the nucleotide framing has read its tables: phase 2 may overwrite them
    const int64_t R0 = sm.s_bound[0][0], R1 = sm.s_bound[1][0];
    const int64_t A = min(sm.s_bound[0][1], total_p), B = min(sm.s_bound[1][1], total_p);
    const int64_t Abase = A & ~(int64_t)15;
    const int nrec = (int)min(R1 - R0 + 1, (int64_t)K23_RCAP + 1);
    const bool slow = sm.s_over != 0 || R1 - R0 + 1 > K23_RCAP || B - Abase > (int64_t)K23_PMAX;
    uint8_t *__restrict__ out = a.out;
    if (slow) {                                       // per residue from global memory; framing below
        for (int64_t r = R0; r <= R1; r++) {
            int32_t naa = a.rec_aa[r];
            if (naa < 0) naa = 0;
            const int64_t f0 = __ldg(a.rec_seg_off + r) + 2 * r;
            const int64_t c0 = __ldg(a.piece_off + f0 + 1) + a.rec_skip[r];
            const int64_t pp = __ldg(a.prot_off + r) + a.rec_pre[r];
            int64_t a_lo = P0 > c0 ? (P0 - c0 + 2) / 3 : 0, a_hi = P0 + tile_len > c0 ? (P0 + tile_len - c0 + 2) / 3 : 0;
            if (a_hi > naa) a_hi = naa;
            for (int64_t x = a_lo + threadIdx.x; x < a_hi; x += NUC_THREADS)
                if (pp + x < total_p) out[pp + x] = k23_residue_generic(a, r, c0 + 3 * x);
        }
    } else {
        reinterpret_cast<uint4 *>(sm.u.p.s_aa)[threadIdx.x] = __ldg(reinterpret_cast<const uint4 *>(a.aa4096h) + threadIdx.x);   // mg_aa_slot order
        int32_t *r_s = sm.u.p.r_s, *r_e = sm.u.p.r_e, *r_q0 = sm.u.p.r_q0;
        for (int i = threadIdx.x; i < nrec + 2; i += NUC_THREADS) {
            if (i < nrec) {
                const int64_t r = R0 + i;
                int32_t naa = a.rec_aa[r];
                if (naa < 0) naa = 0;
                const int64_t f0 = __ldg(a.rec_seg_off + r) + 2 * r;
                const int64_t c0 = __ldg(a.piece_off + f0 + 1) + a.rec_skip[r] - P0;       // tile-relative position of codon 0
                const int64_t pp = __ldg(a.prot_off + r) + a.rec_pre[r] - Abase;            // range-relative position of residue 0
                int64_t a_lo = c0 < 0 ? (-c0 + 2) / 3 : 0, a_hi = tile_len > c0 ? (tile_len - c0 + 2) / 3 : 0;
                if (a_hi > naa) a_hi = naa;
                if (a_lo > a_hi) a_lo = a_hi;
                r_s[i] = (int32_t)(pp + a_lo);
                r_e[i] = (int32_t)(pp + a_hi);
                r_q0[i] = (int32_t)(c0 - 3 * pp);
            } else {
                r_s[i] = BIG; r_e[i] = BIG; r_q0[i] = 0;
            }
        }
        __syncthreads();
        const int n_chunk = (int)((B - Abase + 15) >> 4);
        const uint32_t *__restrict__ s_nib = sm.s_nib;
        const uint8_t *__restrict__ s_aa = sm.u.p.s_aa;
#pragma unroll 1
        for (int cj = threadIdx.x; cj < n_chunk; cj += NUC_THREADS) {
            const int p = cj << 4;
            int R;
            {   // first record whose owned residues end after position p
                int lo = -1, hi = nrec;               // r_e[lo] <= p < r_e[hi]  (r_e[nrec] = BIG)
                while (hi - lo > 1) {
                    const int mid = (lo + hi) >> 1;
                    if (r_e[mid] <= p) lo = mid; else hi = mid;
                }
                R = hi;
            }
            uint32_t bw[4] = {0, 0, 0, 0};
            uint32_t own = 0;                         // chunk bytes that hold residues of this tile
            for (; r_s[R] < p + 16; R++) {
                const int lo = max(r_s[R] - p, 0), hi = min(r_e[R] - p, 16);
                if (hi <= lo) continue;
                const int q = r_q0[R] + 3 * p;        // tile-relative nucleotide position of the codon of chunk position 0
                const int wq = (q >> 3) + 8;          // q >= -45: inside the front slack
                const uint32_t sh = ((uint32_t)q & 7u) << 2;
                uint32_t v[7], n[6];
#pragma unroll
                for (int k = 0; k < 7; k++) v[k] = s_nib[wq + k];
#pragma unroll
                for (int k = 0; k < 6; k++) n[k] = __funnelshift_r(v[k], v[k + 1], sh);
                uint32_t w[4] = {0, 0, 0, 0};
                {
                    constexpr uint32_t M0 = 0x0C00C00Cu, M1 = 0xC00C00C0u, M2 = 0x00C00C00u;   // mg_aa_slot on all 16 codons, see k_emit_prot
                    const uint32_t x0 = n[0] ^ (__funnelshift_r(n[0], n[1], 6) & M0), x1 = n[1] ^ (__funnelshift_r(n[1], n[2], 6) & M1),
                                   x2 = n[2] ^ (__funnelshift_r(n[2], n[3], 6) & M2), x3 = n[3] ^ (__funnelshift_r(n[3], n[4], 6) & M0),
                                   x4 = n[4] ^ (__funnelshift_r(n[4], n[5], 6) & M1), x5 = n[5] ^ ((n[5] >> 6) & M2);
                    n[0] = x0; n[1] = x1; n[2] = x2; n[3] = x3; n[4] = x4; n[5] = x5;
                }
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    const int bit = 12 * k, ww = bit >> 5, s2 = bit & 31;
                    const uint32_t idx = (s2 > 20 ? __funnelshift_r(n[ww], n[ww + 1], s2) : (n[ww] >> s2)) & 0xFFFu;
                    w[k >> 2] |= (uint32_t)s_aa[idx] << ((k & 3) * 8);
                }
                if (q + 3 * hi > tile_len) {          // the codon that straddles the end of the tile: its last bases are not staged
                    const int k = hi - 1;
                    const uint32_t c = k23_residue_generic(a, R0 + R, P0 + q + 3 * k);
                    w[k >> 2] = (w[k >> 2] & ~(0xFFu << ((k & 3) * 8))) | (c << ((k & 3) * 8));
                }
                const uint32_t m = ((1u << hi) - 1u) & ~((1u << lo) - 1u);
                own |= m;
                if (m == 0xFFFFu) { bw[0] = w[0]; bw[1] = w[1]; bw[2] = w[2]; bw[3] = w[3]; }
                else {
#pragma unroll
                    for (int k = 0; k < 4; k++) { const uint32_t mk = expand4(m >> (4 * k)); bw[k] = (bw[k] & ~mk) | (w[k] & mk); }
                }
            }
            const int64_t pos = Abase + p;
            if (pos >= A && pos + 16 <= B) {
                mg_st16(out + pos, bw[0], bw[1], bw[2], bw[3]);
            } else {                                  // chunk shared with a neighbouring tile: only the residues of this one
                for (int k = 0; k < 16; k++)
                    if ((own >> k) & 1u) out[pos + k] = (uint8_t)(bw[k >> 2] >> ((k & 3) * 8));
            }
        }
    }
    __syncthreads();
    // framing bytes of the protein text whose key lies in this tile, four lanes per record (see prot_write_framing)
    if (a.lit) {
        for (int64_t idx = threadIdx.x; idx < (R1 - R0 + 1) * 4; idx += NUC_THREADS) {
            const int64_t r = R0 + (idx >> 2);
            const int sub = (int)(idx & 3);
            const int64_t f0 = __ldg(a.rec_seg_off + r) + 2 * r, f1 = __ldg(a.rec_seg_off + r + 1) + 2 * (r + 1);
            const int64_t start = __ldg(a.piece_off + f0) - P0, sufpos = __ldg(a.piece_off + f1 - 1) - P0;
            const int pre = a.rec_pre[r], suf = a.rec_suf[r];
            int32_t naa = a.rec_aa[r];
            if (naa < 0) naa = 0;
            const int64_t pa = __ldg(a.prot_off + r);
            const uint8_t *src = a.lit + a.rec_lit_off[r];
            if (start >= 0 && start < tile_len) {
                for (int q = sub; q < pre; q += 32) {
                    uint8_t b[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) b[j] = q + 4 * j < pre ? __ldg(src + q + 4 * j) : (uint8_t)0;
#pragma unroll
                    for (int j = 0; j < 8; j++) if (q + 4 * j < pre && pa + q + 4 * j < total_p) out[pa + q + 4 * j] = b[j];
                }
            }
            if (sub == 3 && sufpos >= 0 && sufpos < tile_len)
                for (int q = 0; q < suf; q++) if (pa + pre + naa + q < total_p) out[pa + pre + naa + q] = __ldg(src + pre + q);
        }
    }
}

// ---- host API -----------------------------------------------------------------------------------------------

static int ensure_out(mg_plan *p, int64_t bytes, cudaStream_t st) {
    if (p->out_cap >= bytes) return MG_OK;
    if (p->d_out) MG_CUDA(cudaFreeAsync(p->d_out, st));
    p->d_out = nullptr;
    p->out_cap = 0;
    MG_CUDA(cudaMallocAsync((void **)&p->d_out, bytes, st));
    p->out_cap = bytes;
    return MG_OK;
}

static NucArgs nuc_args(const mg_plan *p, uint8_t *out_dev) {
    const mg_genome *g = p->g;
    NucArgs a;
    a.packed = g->d_packed; a.piece_off = p->d_piece_off; a.piece_src = p->d_piece_src; a.n_piece = p->n_piece;
    a.tile_first = p->d_nuc_tile; a.total_dev = p->d_totals; a.cap = p->nuc_total; a.T = g->total_bases; a.lit = p->d_lit;
    a.exc_pos = g->d_exc_pos; a.exc_byte = g->d_exc_byte; a.n_exc = g->n_exc; a.out = out_dev;
    return a;
}

static ProtArgs prot_args(const mg_plan *p, uint8_t *out_dev) {
    const mg_genome *g = p->g;
    ProtArgs a;
    a.packed = g->d_packed; a.piece_off = p->d_piece_off; a.piece_src = p->d_piece_src; a.rec_seg_off = p->d_rec_seg_off;
    a.prot_off = p->d_prot_off; a.rec_aa = p->d_rec_aa; a.rec_skip = p->d_rec_skip; a.rec_pre = p->d_rec_pre; a.rec_suf = p->d_rec_suf;
    a.rec_lit_off = p->d_rec_lit_off; a.lit = p->n_lit > 0 ? p->d_lit : nullptr; a.n_rec = p->n_rec; a.tile_first = p->d_prot_tile;
    a.total_dev = p->d_totals + 1; a.cap = p->prot_total; a.out = out_dev;
    a.aa4096 = p->own_code ? p->d_aa8192 : g->d_aa4096;             // mg_plan_set_codon_table
    a.aa4096h = p->own_code ? p->d_aa8192 + 4096 : g->d_aa4096h;
    return a;
}

extern "C" int mg_emit_nuc_device(mg_plan *p, uint8_t *out_dev, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    if (const int rc0 = mg_plan_check_prepared(p)) return rc0;
    if (p->nuc_total == 0) return MG_OK;
    MG_REQUIRE(out_dev != nullptr && ((uintptr_t)out_dev & 31) == 0, "out_dev must be a 32-byte aligned device pointer");
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    p->last_stream = st;
    if (mg_emit_mode() == 2) return mg_launch_nuc_stream(p, out_dev, st);
    if (mg_emit_mode() == 1) return mg_launch_nuc_tma(p, out_dev, st);
    k_emit_nuc<<<(unsigned)p->n_nuc_tile, NUC_THREADS, 0, st>>>(nuc_args(p, out_dev));
    MG_LAUNCH_CHECK();
    return MG_OK;
}

extern "C" int mg_emit_prot_device(mg_plan *p, uint8_t *out_dev, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    if (const int rc0 = mg_plan_check_prepared(p)) return rc0;
    if (!p->prot_ready) { mg_set_error("the record pass was deferred (MG_PROT_DEFER): call mg_plan_prepare_prot_async first"); return MG_ESTATE; }
    if (p->prot_total == 0) return MG_OK;
    MG_REQUIRE(out_dev != nullptr && ((uintptr_t)out_dev & 15) == 0, "out_dev must be a 16-byte aligned device pointer");
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    p->last_stream = st;
    k_emit_prot<<<(unsigned)p->n_prot_tile, PROT_THREADS, 0, st>>>(prot_args(p, out_dev));
    MG_LAUNCH_CHECK();
    return MG_OK;
}

// K23: nucleotide text and protein text of one plan in one launch (same buffer rules as the two single calls).
// mg_tune("fuse", 0) makes it the two launches K2 + K3 (A/B and test knob).
static int g_fuse = 1;
void mg_set_fuse(int v) { g_fuse = v; }
extern "C" int mg_emit_nuc_prot_device(mg_plan *p, uint8_t *nuc_out_dev, uint8_t *prot_out_dev, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    if (const int rc0 = mg_plan_check_prepared(p)) return rc0;
    if (!p->prot_ready) { mg_set_error("the record pass was deferred (MG_PROT_DEFER): call mg_plan_prepare_prot_async first"); return MG_ESTATE; }
    if (p->nuc_total == 0) return mg_emit_prot_device(p, prot_out_dev, stream);       // no nucleotide tile: framing-only protein text
    if (p->prot_total == 0) return mg_emit_nuc_device(p, nuc_out_dev, stream);
    if (!g_fuse || mg_emit_mode() != 0) {
        const int rc = mg_emit_nuc_device(p, nuc_out_dev, stream);
        return rc ? rc : mg_emit_prot_device(p, prot_out_dev, stream);
    }
    MG_REQUIRE(nuc_out_dev != nullptr && ((uintptr_t)nuc_out_dev & 31) == 0, "nuc_out_dev must be a 32-byte aligned device pointer");
    MG_REQUIRE(prot_out_dev != nullptr && ((uintptr_t)prot_out_dev & 15) == 0, "prot_out_dev must be a 16-byte aligned device pointer");
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    p->last_stream = st;
    FusedArgs f;
    f.n = nuc_args(p, nuc_out_dev);
    f.p = prot_args(p, prot_out_dev);
    k_emit_nuc_prot<<<(unsigned)p->n_nuc_tile, NUC_THREADS, 0, st>>>(f);
    MG_LAUNCH_CHECK();
    return MG_OK;
}

// ---- all products of a step in ONE launch ----------------------------------------------------------------------------------
// The reference emits, for a transcript, the exon-based transcript text, the CDS text and the protein from the SAME genome
// bases (genome.py:687-710: the CDS children are sub-ranges of the exon children; the protein is the translation of the CDS
// string it has just joined, genome.py:704-707).  As three launches every product fetches those bases from DRAM again
// (config 4, ncu: 368 + 241 + 258 MB read for 183 MB of distinct packed bytes): each launch moves far more than the 126 MB L2
// holds, so nothing survives from one launch to the next.  Here the tiles of up to three jobs -- nucleotide text of plan A
// (exon table), nucleotide text of plan B (CDS table), protein text of plan B -- go into ONE grid in an interleaved order:
// every job advances through its text at the same FRACTIONAL pace (optionally job B a little behind job A and the protein a
// little behind job B: lag).  Both tables list the same transcripts in the same order, so when a CDS tile runs, the exon tiles
// of the same transcripts run in the same wave of CTAs or ran just before, and the 64-byte granules it needs are in L2.
//   order of tile t of job j:  key = floor((2t + 1) * 2^30 / (2 n_j)) + lag_j, ties by (job, tile); k_multi_order turns it
//   into rank -> (job, tile) with closed-form counts (no sort, no search); n_j comes from the text sizes ON THE DEVICE.
#define MULTI_SH 30
#ifndef MULTI_LAG_PPM
#define MULTI_LAG_PPM 0                              // lag between consecutive jobs, in millionths of a text (mg_tune("multi_lag")).  Measured on
                                                     // config 4: lag 0 -> 0.353 ms / 424 MB of DRAM reads, 2 % -> 0.357 ms / 469 MB, 6 % -> 0.375 ms / 789 MB
                                                     // (three launches: 0.378 ms / 868 MB): L2 keeps a line for ~5 % of a launch, and tiles of equal
                                                     // rank run within one wave of each other anyway
#endif
static int g_multi_lag_ppm = MULTI_LAG_PPM;
void mg_set_multi_lag(int ppm) { g_multi_lag_ppm = ppm; }

struct MultiArgs {
    NucArgs a, b;                                    // a.out == nullptr / b.out == nullptr: job absent
    ProtArgs c;                                      // c.out == nullptr: job absent
    int64_t lag[3];
    uint32_t *order;                                 // [capacity] rank -> job << 28 | tile
};

__device__ __forceinline__ int64_t multi_tiles(const int64_t *total_dev, int64_t cap, int64_t tile_bytes, const void *out) {
    if (out == nullptr) return 0;
    const int64_t total = min(__ldg(total_dev), cap);
    return (total + tile_bytes - 1) / tile_bytes;
}
// tiles of a job (n tiles, lag) whose key is < K
__device__ __forceinline__ int64_t multi_count_lt(int64_t K, int64_t n, int64_t lag) {
    const int64_t Kp = K - lag;
    if (Kp <= 0 || n == 0) return 0;
    const int64_t q = (Kp * 2 * n - 1) >> MULTI_SH;
    return min(n, (q + 1) >> 1);
}

__global__ void __launch_bounds__(256) k_multi_order(const __grid_constant__ MultiArgs m) {
    const int64_t n[3] = {multi_tiles(m.a.total_dev, m.a.cap, MG_NUC_TILE, m.a.out), multi_tiles(m.b.total_dev, m.b.cap, MG_NUC_TILE, m.b.out),
                          multi_tiles(m.c.total_dev, m.c.cap, MG_PROT_TILE, m.c.out)};
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int j = 0;
    if (t >= n[0]) { t -= n[0]; j = 1; if (t >= n[1]) { t -= n[1]; j = 2; if (t >= n[2]) return; } }
    const int64_t K = (((2 * t + 1) << MULTI_SH) / (2 * n[j])) + m.lag[j];
    int64_t rank = t;
#pragma unroll
    for (int jj = 0; jj < 3; jj++)
        if (jj != j) rank += multi_count_lt(jj < j ? K + 1 : K, n[jj], m.lag[jj]);
    m.order[rank] = ((uint32_t)j << 28) | (uint32_t)t;
}

__global__ void __launch_bounds__(NUC_THREADS, NUC_MINB) k_emit_multi(const __grid_constant__ MultiArgs m) {
    __shared__ union { NucSmem n; ProtSmem p; } sm;
    const int64_t na = multi_tiles(m.a.total_dev, m.a.cap, MG_NUC_TILE, m.a.out), nb = multi_tiles(m.b.total_dev, m.b.cap, MG_NUC_TILE, m.b.out),
                  nc = multi_tiles(m.c.total_dev, m.c.cap, MG_PROT_TILE, m.c.out);
    if (blockIdx.x >= na + nb + nc) return;
    const uint32_t o = __ldg(m.order + blockIdx.x);
    const int64_t tile = o & 0x0FFFFFFFu;
    const uint32_t job = o >> 28;
    if (job == 0) nuc_tile<false, NUC_CAP>(m.a, sm.n, tile, min(__ldg(m.a.total_dev), m.a.cap));
    else if (job == 1) nuc_tile<false, NUC_CAP>(m.b, sm.n, tile, min(__ldg(m.b.total_dev), m.b.cap));
    else prot_tile(m.c, sm.p, tile, min(__ldg(m.c.total_dev), m.c.cap));
}

// Nucleotide text of plan `pa` (-> out_a), nucleotide text of plan `pb` (-> out_b_nuc) and protein text of `pb` (-> out_b_prot) in
// one launch; any output pointer may be NULL (that product is skipped; pa / pb may then be NULL too).  Both plans must be
// prepared (mg_plan_prepare or mg_plan_prepare_async, the latter on this stream or joined with it) and belong to one genome.
extern "C" int mg_emit_products_device(mg_plan *pa, uint8_t *out_a, mg_plan *pb, uint8_t *out_b_nuc, uint8_t *out_b_prot, void *stream) {
    const bool ja = pa && out_a && pa->nuc_total > 0, jb = pb && out_b_nuc && pb->nuc_total > 0, jc = pb && out_b_prot && pb->prot_total > 0;
    MG_REQUIRE(!out_a || pa, "out_a given without a plan");
    MG_REQUIRE((!out_b_nuc && !out_b_prot) || pb, "out_b given without a plan");
    if (pa && out_a) { if (const int rc0 = mg_plan_check_prepared(pa)) return rc0; }
    if (pb && (out_b_nuc || out_b_prot)) { if (const int rc0 = mg_plan_check_prepared(pb)) return rc0; }
    if (jc && !pb->prot_ready) { mg_set_error("the record pass was deferred (MG_PROT_DEFER): call mg_plan_prepare_prot_async first"); return MG_ESTATE; }
    if (!ja && !jb && !jc) return MG_OK;
    MG_REQUIRE(!ja || ((uintptr_t)out_a & 31) == 0, "out_a must be a 32-byte aligned device pointer");
    MG_REQUIRE(!jb || ((uintptr_t)out_b_nuc & 31) == 0, "out_b_nuc must be a 32-byte aligned device pointer");
    MG_REQUIRE(!jc || ((uintptr_t)out_b_prot & 15) == 0, "out_b_prot must be a 16-byte aligned device pointer");
    MG_REQUIRE(!(ja && (jb || jc)) || pa->g == pb->g, "both plans must belong to the same genome");
    mg_plan *owner = ja ? pa : pb;
    MG_CUDA(cudaSetDevice(owner->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t cap = (ja ? pa->n_nuc_tile : 0) + (jb ? pb->n_nuc_tile : 0) + (jc ? pb->n_prot_tile : 0);
    MG_REQUIRE(cap < (1ll << 28), "more than 2^28 tiles in one launch");
    if (owner->order_cap < cap) {
        const int rc0 = mg_refuse_growth_in_capture(st, "mg_emit_products_device (first emit led by this plan, or a larger grid)");
        if (rc0) return rc0;
    }
    MultiArgs m;
    memset(&m, 0, sizeof(m));
    if (ja) { m.a = nuc_args(pa, out_a); pa->last_stream = st; }
    if (jb) m.b = nuc_args(pb, out_b_nuc);
    if (jc) m.c = prot_args(pb, out_b_prot);
    if (jb || jc) pb->last_stream = st;
    const int64_t lag = ((int64_t)g_multi_lag_ppm << MULTI_SH) / 1000000;
    m.lag[0] = 0; m.lag[1] = ja ? lag : 0; m.lag[2] = m.lag[1] + (jb ? lag : 0);
    if (owner->order_cap < cap) {
        void *d = nullptr;
        MG_CUDA(cudaMallocAsync(&d, cap * sizeof(uint32_t), st));
        owner->owned.push_back(d);
        owner->d_order = (uint32_t *)d;
        owner->order_cap = cap;
    }
    m.order = owner->d_order;
    k_multi_order<<<(unsigned)((cap + 255) / 256), 256, 0, st>>>(m);
    MG_LAUNCH_CHECK();
    k_emit_multi<<<(unsigned)cap, NUC_THREADS, 0, st>>>(m);
    MG_LAUNCH_CHECK();
    return MG_OK;
}

// Device text -> caller's host buffer.  Page-locked destination: one stream-ordered copy at the PCIe rate.  Pageable destination
// (a numpy array, a Python bytes object): a pageable cudaMemcpy runs at ~10 GB/s, so the text goes through two page-locked
// 32 MB staging buffers instead -- the copy engine fills one while host threads empty the other into the destination -- and
// the call returns when the text is complete.
static int copy_text_to_host(mg_plan *p, uint8_t *out_host, const uint8_t *d_src, int64_t n, cudaStream_t st) {
    cudaPointerAttributes at;
    const bool pinned = cudaPointerGetAttributes(&at, out_host) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();
    const int64_t CH = 32ll << 20;
    if (pinned || n < 2 * CH) {
        MG_CUDA(cudaMemcpyAsync(out_host, d_src, n, cudaMemcpyDeviceToHost, st));
        return MG_OK;
    }
    mg_genome *g = p->g;
    int rc = mg_ensure_pin(g, 2 * CH);
    if (rc) return rc;
    uint8_t *pin[2] = {g->h_pin, g->h_pin + CH};
    cudaEvent_t ev[2];
    MG_CUDA(cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming));
    MG_CUDA(cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming));
    const int64_t nch = (n + CH - 1) / CH;
    cudaError_t e = cudaMemcpyAsync(pin[0], d_src, std::min(CH, n), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaEventRecord(ev[0], st);
    for (int64_t k = 0; k < nch && e == cudaSuccess; k++) {
        const int64_t off = k * CH, m = std::min(CH, n - off);
        if (k + 1 < nch) {                               // its buffer was emptied by the host in the previous iteration
            e = cudaMemcpyAsync(pin[(k + 1) & 1], d_src + off + CH, std::min(CH, n - off - CH), cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaEventRecord(ev[(k + 1) & 1], st);
            if (e != cudaSuccess) break;
        }
        e = cudaEventSynchronize(ev[k & 1]);
        if (e != cudaSuccess) break;
        mg_parallel_copy(pin[k & 1], out_host + off, m);
    }
    cudaEventDestroy(ev[0]);
    cudaEventDestroy(ev[1]);
    if (e != cudaSuccess) { mg_set_error("device -> host text copy failed: %s", cudaGetErrorString(e)); return MG_ECUDA; }
    return MG_OK;
}

extern "C" int mg_emit_nuc_host(mg_plan *p, uint8_t *out_host, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    if (const int rc0 = mg_plan_check_prepared(p)) return rc0;
    if (!p->totals_known) { int rc0 = mg_plan_totals(p, nullptr, nullptr, stream); if (rc0) return rc0; }
    if (p->nuc_total == 0) return MG_OK;
    MG_REQUIRE(out_host != nullptr, "out_host is NULL");
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = ensure_out(p, (p->nuc_total + 31) / 32 * 32, st);
    if (rc) return rc;
    rc = mg_emit_nuc_device(p, p->d_out, stream);
    if (rc) return rc;
    return copy_text_to_host(p, out_host, p->d_out, p->nuc_total, st);
}

// K23 into two library-owned device buffers, then both texts to the host (stream-ordered; mg_stream_sync before reading)
extern "C" int mg_emit_nuc_prot_host(mg_plan *p, uint8_t *nuc_out_host, uint8_t *prot_out_host, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    if (const int rc0 = mg_plan_check_prepared(p)) return rc0;
    if (!p->totals_known) { int rc0 = mg_plan_totals(p, nullptr, nullptr, stream); if (rc0) return rc0; }
    if (p->nuc_total == 0 && p->prot_total == 0) return MG_OK;
    MG_REQUIRE((nuc_out_host != nullptr || p->nuc_total == 0) && (prot_out_host != nullptr || p->prot_total == 0), "output buffer is NULL");
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nn = (p->nuc_total + 31) / 32 * 32, np = (p->prot_total + 31) / 32 * 32;
    int rc = ensure_out(p, nn + np + 32, st);
    if (rc) return rc;
    rc = mg_emit_nuc_prot_device(p, p->d_out, p->d_out + nn, stream);
    if (rc) return rc;
    if (p->nuc_total) { rc = copy_text_to_host(p, nuc_out_host, p->d_out, p->nuc_total, st); if (rc) return rc; }
    if (p->prot_total) rc = copy_text_to_host(p, prot_out_host, p->d_out + nn, p->prot_total, st);
    return rc;
}

// mg_emit_products_device into library-owned device buffers, then the texts to the host (stream-ordered)
extern "C" int mg_emit_products_host(mg_plan *pa, uint8_t *out_a_host, mg_plan *pb, uint8_t *out_b_nuc_host, uint8_t *out_b_prot_host,
                                     void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *da = nullptr, *dbn = nullptr, *dbp = nullptr;
    if (pa && out_a_host) {
        if (const int rc0 = mg_plan_check_prepared(pa)) return rc0;
        if (!pa->totals_known) { int rc0 = mg_plan_totals(pa, nullptr, nullptr, stream); if (rc0) return rc0; }
        MG_CUDA(cudaSetDevice(pa->device));
        int rc = ensure_out(pa, (pa->nuc_total + 31) / 32 * 32 + 32, st);
        if (rc) return rc;
        da = pa->d_out;
    }
    int64_t nn = 0;
    if (pb && (out_b_nuc_host || out_b_prot_host)) {
        if (const int rc0 = mg_plan_check_prepared(pb)) return rc0;
        if (!pb->totals_known) { int rc0 = mg_plan_totals(pb, nullptr, nullptr, stream); if (rc0) return rc0; }
        MG_CUDA(cudaSetDevice(pb->device));
        nn = out_b_nuc_host ? (pb->nuc_total + 31) / 32 * 32 : 0;
        int rc = ensure_out(pb, nn + (pb->prot_total + 31) / 32 * 32 + 32, st);
        if (rc) return rc;
        if (out_b_nuc_host) dbn = pb->d_out;
        if (out_b_prot_host) dbp = pb->d_out + nn;
    }
    int rc = mg_emit_products_device(pa, da, pb, dbn, dbp, stream);
    if (rc) return rc;
    if (da && pa->nuc_total) { rc = copy_text_to_host(pa, out_a_host, da, pa->nuc_total, st); if (rc) return rc; }
    if (dbn && pb->nuc_total) { rc = copy_text_to_host(pb, out_b_nuc_host, dbn, pb->nuc_total, st); if (rc) return rc; }
    if (dbp && pb->prot_total) rc = copy_text_to_host(pb, out_b_prot_host, dbp, pb->prot_total, st);
    return rc;
}

extern "C" int mg_emit_prot_host(mg_plan *p, uint8_t *out_host, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    if (const int rc0 = mg_plan_check_prepared(p)) return rc0;
    if (!p->totals_known) { int rc0 = mg_plan_totals(p, nullptr, nullptr, stream); if (rc0) return rc0; }
    if (p->prot_total == 0) return MG_OK;
    MG_REQUIRE(out_host != nullptr, "out_host is NULL");
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = ensure_out(p, (p->prot_total + 31) / 32 * 32, st);
    if (rc) return rc;
    rc = mg_emit_prot_device(p, p->d_out, stream);
    if (rc) return rc;
    return copy_text_to_host(p, out_host, p->d_out, p->prot_total, st);
}
