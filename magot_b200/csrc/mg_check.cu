// mg_check.cu -- gene-model check of a prepared plan (mg_plan_check*): start and stop codons, in-frame stops, reading frame,
// ambiguous codons, GC / GC3, codon usage and splice-site classes per record.  Semantics: include/magot_b200.h.
//
// Four launches on one stream, no host round trip:
//   k_check_records   thread per record: skip, rem, n_codons, start and stop codon; zeroes the accumulators (and the 64 bins
//                     of records whose codons span more than one tile);
//   k_check_codons    flat over the nucleotide text in the plan's 32 KB tiles (the tile table K2 uses, no new scan): a codon
//                     belongs to the tile that holds its first base.  A lane owns 48 text positions (at most 16 codon starts of
//                     one record), gathers their 48 nibbles from the packed plane with K3's window (one one-sided mask per
//                     piece), and classifies each codon with one shared-memory look-up.  Sums go to per-record slots in shared
//                     memory; a record whose codons all lie in the tile is stored plainly, one that straddles tiles is added
//                     with one global atomic per field and tile.  A tile whose pieces overflow the staging reads each codon
//                     through the generic global gather (correct, slow); records are taken in batches of CHK_RCAP;
//   k_check_junctions thread per caller segment: two dinucleotides from the forward or the reverse plane;
//   k_check_final     thread per record: first stop, terminal stop, flags.
// Every genome index is 64-bit; text positions inside a tile are 32-bit and relative to the tile.
#include <algorithm>
#include <climits>
#include <cstring>
#include "mg_common.cuh"
#include "mg_gather.cuh"
#include "mg_emit_common.cuh"

#define CHK_THREADS 256
#define CHK_RCAP 64                                   // records staged per batch (a 32 KB tile of config 4 holds ~30)
#define CHK_PCAP 768                                  // pieces staged per tile (~200 in config 4)
#define CHK_SPAN 48                                   // text positions per lane: at most 16 codon starts
#define CHK_NSPAN ((MG_NUC_TILE + CHK_SPAN - 1) / CHK_SPAN)
#define CHK_BIG (1 << 30)
#define CHK_AMBIG 0x80u                               // class entry: bits 0-5 codon index, bit 6 stop, bit 7 ambiguous
#define CHK_STOP 0x40u

static_assert(sizeof(mg_cds_check) == 56, "mg_cds_check layout (include/magot_b200.h)");

struct ChkArgs {
    const uint32_t *packed;
    const int64_t *piece_off, *piece_src, *rec_seg_off;
    const int64_t *tile_first, *total_dev;
    int64_t cap, n_rec;
    uint64_t stop_mask;
    mg_cds_check *rec;
    uint32_t *counts;
};

// 12-bit nibble triplet (first base lowest) -> class entry
__device__ __forceinline__ uint32_t chk_class(uint32_t c, uint64_t stop_mask) {
    if (c & 0x888u) return CHK_AMBIG;
    const uint32_t idx = ((c & 3u) << 4) | (((c >> 4) & 3u) << 2) | ((c >> 8) & 3u);
    return idx | (((stop_mask >> idx) & 1u) ? CHK_STOP : 0u);
}

// G/C among the three bases of codon index idx (b2 in bits 0-1, b1 in 2-3, b0 in 4-5; C = 1 and G = 2 are the codes whose two
// bits differ) and whether the third base is G/C
__device__ __forceinline__ uint32_t chk_gc(uint32_t idx) { return __popc((idx ^ (idx >> 1)) & 0x15u); }
__device__ __forceinline__ uint32_t chk_gc3(uint32_t idx) { return (idx ^ (idx >> 1)) & 1u; }

// the nibble triplet of the codon at nucleotide-text position S of record r, through the record's pieces in global memory
__device__ __noinline__ uint32_t chk_codon_generic(const ChkArgs &a, int64_t r, int64_t S) {
    const int64_t f0 = __ldg(a.rec_seg_off + r) + 2 * r, f1 = __ldg(a.rec_seg_off + r + 1) + 2 * (r + 1);
    const int64_t j = mg_search_le(a.piece_off, f0 + 1, f1 - 1, S);
    uint64_t acc[3];
    mg_gather_nib(a.packed, a.piece_off, a.piece_src, j, S, 3, acc);
    return (uint32_t)acc[0] & 0xFFFu;
}

// first codon of a record's codon range spans [c_first, c_last + 3); it is owned by one tile when both ends start in it
__device__ __forceinline__ bool chk_one_tile(int64_t c_first, int64_t c_last) {
    return c_first / MG_NUC_TILE == c_last / MG_NUC_TILE;
}

__global__ void __launch_bounds__(256) k_check_records(const __grid_constant__ ChkArgs a, const int8_t *__restrict__ rec_phase, int use_phase) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= a.n_rec) return;
    const int64_t f0 = __ldg(a.rec_seg_off + r) + 2 * r, f1 = __ldg(a.rec_seg_off + r + 1) + 2 * (r + 1);
    const int64_t ns = __ldg(a.piece_off + f0 + 1), len = __ldg(a.piece_off + f1 - 1) - ns;
    int skip = use_phase && rec_phase ? rec_phase[r] : 0;
    if (skip < 0 || skip > 2) skip = 0;
    const int64_t L = len - skip;
    const int64_t ncod = L > 0 ? L / 3 : 0;
    const int rem = L > 0 ? (int)(L % 3) : 0;
    uint32_t sc = 0xFFu, ec = 0xFFu;
    if (ncod > 0) {
        uint64_t acc[3];
        mg_gather_nib(a.packed, a.piece_off, a.piece_src, f0 + 1, ns + skip, 3, acc);
        uint32_t e = chk_class((uint32_t)acc[0] & 0xFFFu, a.stop_mask);
        sc = (e & CHK_AMBIG) ? 0xFFu : (e & 63u);
        const int64_t S = ns + skip + 3 * (ncod - 1);
        e = chk_class(chk_codon_generic(a, r, S), a.stop_mask);
        ec = (e & CHK_AMBIG) ? 0xFFu : (e & 63u);
    }
    mg_cds_check c;
    c.nuc_len = len;
    c.gc = 0;
    c.n_codons = (int32_t)ncod;
    c.n_ambig = 0;
    c.n_stop = 0;
    c.first_stop = INT_MAX;                           // k_check_codons takes the minimum; k_check_final turns "none" into -1
    c.gc3 = 0;
    c.n_junction = 0;
    c.n_noncanonical = 0;
    c.flags = 0;
    c.skip = (int8_t)skip;
    c.rem = (int8_t)rem;
    c.start_codon = (uint8_t)sc;
    c.stop_codon = (uint8_t)ec;
    c.pad = 0;
    a.rec[r] = c;
    // bins of a record that k_check_codons does not store whole: it adds to them, or (no codon) never touches them
    if (a.counts && !(ncod > 0 && chk_one_tile(ns + skip, ns + skip + 3 * (ncod - 1)))) {
        uint4 *b = reinterpret_cast<uint4 *>(a.counts + 64 * r);
#pragma unroll
        for (int k = 0; k < 16; k++) b[k] = make_uint4(0, 0, 0, 0);
    }
}

// record that owns piece `pc` (F(r) = rec_seg_off[r] + 2r <= pc < F(r+1)): 32-ary search by one warp
__device__ __forceinline__ int64_t chk_record_of_piece(const int64_t *__restrict__ rec_seg_off, int64_t n_rec, int64_t pc, int lane) {
    int64_t lo = 0, hi = n_rec;                       // answer in [lo, hi)
    while (hi - lo > 1) {
        const int64_t step = (hi - lo + 31) / 32;
        const int64_t r = lo + (int64_t)lane * step;
        const bool le = r < hi && __ldg(rec_seg_off + r) + 2 * r <= pc;
        const unsigned int b = __ballot_sync(0xffffffffu, le);
        const int k = 31 - __clz(b);
        lo = lo + (int64_t)k * step;
        hi = min(hi, lo + step);
    }
    return lo;
}

template <bool COUNTS>
struct ChkSmem {
    __align__(16) uint8_t cls[4096];                 // class entry of nibble triplet c at mg_aa_slot(c) (one wavefront a look-up)
    int64_t s_base[CHK_PCAP + 2];                    // genome index of the piece's base at tile position 0
    int32_t s_rel[CHK_PCAP + 3];                     // piece i covers tile positions [s_rel[i], s_rel[i+1]) (clamped to +-CHK_BIG)
    int32_t r_s[CHK_RCAP + 1], r_e[CHK_RCAP + 1];    // codon starts of the batch's records in this tile: r_s, r_s + 3, ... < r_e
    int32_t r_k0[CHK_RCAP];                          // codon index of r_s
    uint8_t r_flag[CHK_RCAP];                        // bit 0: codons in this tile, bit 1: all of the record's codons
    uint32_t a_ambig[CHK_RCAP], a_stop[CHK_RCAP], a_gc[CHK_RCAP], a_gc3[CHK_RCAP];
    int32_t a_first[CHK_RCAP];
    uint32_t bins[COUNTS ? CHK_RCAP * 64 : 1];
    int64_t s_rec[2];
};

#define CHK_MINB 4
template <bool COUNTS>
__global__ void __launch_bounds__(CHK_THREADS, CHK_MINB) k_check_codons(const __grid_constant__ ChkArgs a) {
    const int64_t total = min(__ldg(a.total_dev), a.cap);
    const int64_t tile = blockIdx.x;
    const int64_t P0 = tile * MG_NUC_TILE;
    if (P0 >= total) return;
    __shared__ ChkSmem<COUNTS> sm;
    const int tile_len = (int)min((int64_t)MG_NUC_TILE, total - P0);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t pf = __ldg(a.tile_first + tile), pl = __ldg(a.tile_first + tile + 1);   // pieces of the first and the next tile's first byte
    if (wid < 2) {
        const int64_t r = chk_record_of_piece(a.rec_seg_off, a.n_rec, wid ? pl : pf, lane);
        if (lane == 0) sm.s_rec[wid] = r;
    }
    for (int c = threadIdx.x; c < 4096; c += CHK_THREADS) sm.cls[mg_aa_slot(c)] = (uint8_t)chk_class(c, a.stop_mask);
    const int64_t npc64 = pl - pf + 1;
    const bool fast = npc64 <= CHK_PCAP;
    if (fast) {
        const int npc = (int)npc64;
        for (int i = threadIdx.x; i <= npc + 1; i += CHK_THREADS) {
            if (i <= npc) {
                const int64_t off = __ldg(a.piece_off + pf + i) - P0;
                sm.s_rel[i] = (int32_t)max(min(off, (int64_t)CHK_BIG), -(int64_t)CHK_BIG);
                sm.s_base[i] = i < npc ? (int64_t)((uint64_t)__ldg(a.piece_src + pf + i) & MG_SRC_MASK) - off : 0;
            } else {
                sm.s_rel[i] = CHK_BIG;
            }
        }
    }
    __syncthreads();
    const int64_t R0 = sm.s_rec[0], nrec = sm.s_rec[1] - R0 + 1;
    for (int64_t b0 = 0; b0 < nrec; b0 += CHK_RCAP) {
        const int nb = (int)min((int64_t)CHK_RCAP, nrec - b0);
        for (int i = threadIdx.x; i <= nb; i += CHK_THREADS) {
            if (i == nb) { sm.r_s[i] = sm.r_e[i] = CHK_BIG; continue; }
            const int64_t r = R0 + b0 + i;
            const int64_t f0 = __ldg(a.rec_seg_off + r) + 2 * r;
            const int64_t ncod = a.rec[r].n_codons;
            const int64_t ns = __ldg(a.piece_off + f0 + 1);
            const int64_t c0 = ns + a.rec[r].skip - P0;       // tile position of codon 0
            int64_t k_hi = tile_len > c0 ? (tile_len - c0 + 2) / 3 : 0, k_lo = c0 >= 0 ? 0 : (-c0 + 2) / 3;
            if (k_hi > ncod) k_hi = ncod;
            if (k_lo > k_hi) k_lo = k_hi;
            if (k_hi > k_lo) {
                sm.r_s[i] = (int32_t)(c0 + 3 * k_lo);
                sm.r_e[i] = (int32_t)(c0 + 3 * k_hi);
                sm.r_flag[i] = 1 | (chk_one_tile(c0 + P0, c0 + P0 + 3 * (ncod - 1)) ? 2 : 0);
            } else {                                   // no codon here: an empty range where the record's payload starts
                const int32_t v = (int32_t)max(min(ns - P0, (int64_t)tile_len + 3), (int64_t)0);
                sm.r_s[i] = sm.r_e[i] = v;
                sm.r_flag[i] = 0;
            }
            sm.r_k0[i] = (int32_t)k_lo;
            sm.a_ambig[i] = sm.a_stop[i] = sm.a_gc[i] = sm.a_gc3[i] = 0;
            sm.a_first[i] = INT_MAX;
        }
        if (COUNTS)
            for (int i = threadIdx.x; i < nb * 64; i += CHK_THREADS) sm.bins[i] = 0;
        __syncthreads();
#pragma unroll 1
        for (int cj = threadIdx.x; cj < CHK_NSPAN; cj += CHK_THREADS) {
            const int p = cj * CHK_SPAN;
            if (p >= tile_len) break;
            int R;
            {   // first record of the batch whose codon starts end after p
                int lo = -1, hi = nb;                  // r_e[lo] <= p < r_e[hi]  (r_e[nb] = CHK_BIG)
                while (hi - lo > 1) {
                    const int mid = (lo + hi) >> 1;
                    if (sm.r_e[mid] <= p) lo = mid; else hi = mid;
                }
                R = hi;
            }
            for (; sm.r_s[R] < p + CHK_SPAN; R++) {
                const int rs = sm.r_s[R];
                const int lo_pos = max(p, rs);
                const int q = rs + (lo_pos - rs + 2) / 3 * 3;          // first codon start of R in [p, p + 48)
                const int hi_pos = min(p + CHK_SPAN, sm.r_e[R]);
                if (q >= hi_pos) continue;
                const int n = (hi_pos - q + 2) / 3;                    // 1..16 codons
                const int k0 = sm.r_k0[R] + (q - rs) / 3;
                const int64_t r = R0 + b0 + R;
                uint32_t w[6] = {0, 0, 0, 0, 0, 0};
                if (fast) {
                    // the 48 nibbles from the tile's staged pieces, left to right, each overwriting the window from its first
                    // nibble on (K3's gather); nibbles at or past the tile end are not staged
                    const int need_hi = min(q + 3 * n, tile_len);
                    int X;
                    {
                        int lo = 0, hi = (int)npc64 + 1;   // last piece with s_rel <= q
                        while (hi - lo > 1) {
                            const int mid = (lo + hi) >> 1;
                            if (sm.s_rel[mid] <= q) lo = mid; else hi = mid;
                        }
                        X = lo;
                    }
#pragma unroll 1
                    for (int j = X; sm.s_rel[j] < need_hi; j++) {
                        const int c = sm.s_rel[j] - q;
                        if (sm.s_rel[j + 1] - q <= c) continue;        // empty piece
                        const int64_t g = sm.s_base[j] + q;
                        const uint32_t *pp = a.packed + (g >> 3);
                        const uint32_t sh = ((uint32_t)g & 7u) << 2;
                        uint32_t v[7];
#pragma unroll
                        for (int k = 0; k < 7; k++) v[k] = ld_pk(pp + k);
#pragma unroll
                        for (int k = 0; k < 6; k++) {
                            const uint32_t keep = low_nibbles(c - 8 * k);
                            w[k] = (w[k] & keep) | (__funnelshift_r(v[k], v[k + 1], sh) & ~keep);
                        }
                    }
                }
                uint32_t amb = 0, stp = 0, gc = 0, gc3 = 0;
                int first = INT_MAX;
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    if (k >= n) break;
                    uint32_t c12;
                    if (fast && q + 3 * k + 3 <= tile_len) {
                        const int bit = 12 * k, ww = bit >> 5, s2 = bit & 31;
                        c12 = (s2 > 20 ? __funnelshift_r(w[ww], w[ww + 1], s2) : (w[ww] >> s2)) & 0xFFFu;
                    } else {                                   // the codon that straddles the tile end, or a tile that did not stage
                        c12 = chk_codon_generic(a, r, P0 + q + 3 * k);
                    }
                    const uint32_t e = sm.cls[mg_aa_slot(c12)];
                    if (e & CHK_AMBIG) { amb++; continue; }
                    const uint32_t idx = e & 63u;
                    if (e & CHK_STOP) { stp++; first = min(first, k0 + k); }
                    gc += chk_gc(idx);
                    gc3 += chk_gc3(idx);
                    if (COUNTS) atomicAdd(&sm.bins[R * 64 + idx], 1u);
                }
                if (amb) atomicAdd(&sm.a_ambig[R], amb);
                if (stp) { atomicAdd(&sm.a_stop[R], stp); atomicMin(&sm.a_first[R], first); }
                if (gc) atomicAdd(&sm.a_gc[R], gc);
                if (gc3) atomicAdd(&sm.a_gc3[R], gc3);
            }
        }
        __syncthreads();
        // flush: plain stores for a record whose codons all lie in this tile, global atomics for one that straddles tiles
        for (int i = threadIdx.x; i < nb; i += CHK_THREADS) {
            const uint8_t fl = sm.r_flag[i];
            if (!(fl & 1)) continue;
            mg_cds_check *c = a.rec + R0 + b0 + i;
            if (fl & 2) {
                c->n_ambig = (int32_t)sm.a_ambig[i];
                c->n_stop = (int32_t)sm.a_stop[i];
                c->first_stop = sm.a_first[i];
                c->gc = sm.a_gc[i];
                c->gc3 = (int32_t)sm.a_gc3[i];
            } else {
                if (sm.a_ambig[i]) atomicAdd(&c->n_ambig, (int32_t)sm.a_ambig[i]);
                if (sm.a_stop[i]) { atomicAdd(&c->n_stop, (int32_t)sm.a_stop[i]); atomicMin(&c->first_stop, sm.a_first[i]); }
                if (sm.a_gc[i]) atomicAdd(reinterpret_cast<unsigned long long *>(&c->gc), (unsigned long long)sm.a_gc[i]);
                if (sm.a_gc3[i]) atomicAdd(&c->gc3, (int32_t)sm.a_gc3[i]);
            }
        }
        if (COUNTS) {
            for (int i = threadIdx.x; i < nb * 64; i += CHK_THREADS) {
                const uint8_t fl = sm.r_flag[i >> 6];
                if (!(fl & 1)) continue;
                uint32_t *dst = a.counts + 64 * (R0 + b0) + i;
                const uint32_t v = sm.bins[i];
                if (fl & 2) *dst = v;
                else if (v) atomicAdd(dst, v);
            }
        }
        __syncthreads();                               // the next batch re-stages the record slots
    }
}

// splice-site class of the junction after caller segment e (include/magot_b200.h)
__global__ void __launch_bounds__(256) k_check_junctions(int64_t n_seg, int64_t n_rec, const int64_t *__restrict__ rec_seg_off,
                                                         const int32_t *__restrict__ seg_contig, const int64_t *__restrict__ seg_start,
                                                         const int64_t *__restrict__ seg_end, const int8_t *__restrict__ seg_strand,
                                                         const int64_t *__restrict__ contig_len, const int64_t *__restrict__ contig_base,
                                                         int64_t n_contigs, int64_t two_T, const uint32_t *__restrict__ packed,
                                                         mg_cds_check *rec, int8_t *__restrict__ junction) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= n_seg) return;
    const int64_t r = mg_search_le(rec_seg_off, 0, n_rec, e);
    int cls = 0;
    if (e + 1 < __ldg(rec_seg_off + r + 1)) {
        int64_t lo[2], hi[2];
        int32_t c[2];
        bool minus[2];
        for (int k = 0; k < 2; k++) {                  // contig[start-1:end] with Python slice semantics, as the plan kernels
            c[k] = __ldg(seg_contig + e + k);
            minus[k] = __ldg(seg_strand + e + k) != 0;
            lo[k] = hi[k] = 0;
            if (c[k] >= 0 && c[k] < n_contigs) {
                const int64_t L = __ldg(contig_len + c[k]);
                int64_t i = __ldg(seg_start + e + k) - 1, j = __ldg(seg_end + e + k);
                if (i < 0) { i += L; if (i < 0) i = 0; } else if (i > L) i = L;
                if (j < 0) { j += L; if (j < 0) j = 0; } else if (j > L) j = L;
                lo[k] = i;
                hi[k] = j > i ? j : i;
            }
        }
        if (hi[0] > lo[0] && hi[1] > lo[1] && c[0] == c[1] && minus[0] == minus[1]) {
            const int64_t cb = __ldg(contig_base + c[0]);
            int64_t gd = -1, ga = -1;                  // donor / acceptor dinucleotide, read 5'->3' on the transcript strand
            if (!minus[0] && lo[1] - hi[0] >= 4) {
                gd = cb + hi[0];
                ga = cb + lo[1] - 2;
            } else if (minus[0] && lo[0] - hi[1] >= 4) {   // the reverse complement of forward [x, x+2) is reverse-plane [2T-x-2, 2T-x)
                gd = two_T - cb - lo[0];
                ga = two_T - cb - hi[1] - 2;
            }
            if (gd >= 0) {
                const uint32_t d = (uint32_t)mg_ld_nib16(packed, gd) & 0xFFu, x = (uint32_t)mg_ld_nib16(packed, ga) & 0xFFu;
                cls = 4;
                if (!((d | x) & 0x88u)) {
                    const uint32_t dd = (d & 3u) * 4 + ((d >> 4) & 3u), aa = (x & 3u) * 4 + ((x >> 4) & 3u);
                    if (dd == 11 && aa == 2) cls = 1;                  // GT-AG
                    else if (dd == 9 && aa == 2) cls = 2;              // GC-AG
                    else if (dd == 3 && aa == 1) cls = 3;              // AT-AC
                }
            }
        }
    }
    if (junction) junction[e] = (int8_t)cls;
    if (cls) {
        atomicAdd(&rec[r].n_junction, 1);
        if (cls == 4) atomicAdd(&rec[r].n_noncanonical, 1);
    }
}

__global__ void __launch_bounds__(256) k_check_final(int64_t n_rec, uint64_t stop_mask, uint64_t start_mask, mg_cds_check *rec) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    mg_cds_check c = rec[r];
    const bool terminal = c.n_codons > 0 && c.stop_codon != 0xFF && ((stop_mask >> c.stop_codon) & 1);
    int f = 0;
    if (c.start_codon == 0xFF || !((start_mask >> c.start_codon) & 1)) f |= MG_CHK_NO_START;
    if (!terminal) f |= MG_CHK_NO_STOP;
    if (c.n_stop - (terminal ? 1 : 0) > 0) f |= MG_CHK_INTERNAL_STOP;
    if (c.rem) f |= MG_CHK_PARTIAL_CODON;
    if (c.n_noncanonical) f |= MG_CHK_NONCANONICAL_SPLICE;
    if (c.n_ambig) f |= MG_CHK_AMBIGUOUS;
    if (c.n_codons == 0) f |= MG_CHK_EMPTY;
    rec[r].first_stop = c.first_stop == INT_MAX ? -1 : c.first_stop;
    rec[r].flags = f;
}

// ---- host API -----------------------------------------------------------------------------------------------

int mg_start_mask(const mg_plan *p, const uint8_t *start64, uint64_t *start_mask) {
    uint64_t m = 0;
    if (!start64) {
        m = 1ull << 14;                                // ATG: 16*0 + 4*3 + 2 (A=0 C=1 G=2 T=3)
    } else {
        for (int c = 0; c < 64; c++) {
            if (!start64[c]) continue;
            if ((p->stop_mask >> c) & 1) {
                mg_set_error("start codon %c%c%c is a stop codon of this genetic code", "ACGT"[c >> 4], "ACGT"[(c >> 2) & 3], "ACGT"[c & 3]);
                return MG_EINVAL;
            }
            m |= 1ull << c;
        }
        MG_REQUIRE(m != 0, "start64 flags no start codon");
    }
    *start_mask = m;
    return MG_OK;
}

static int check_args(mg_plan *p, int flags, const uint8_t *start64, uint64_t *start_mask) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    MG_REQUIRE((flags & ~MG_PROT_USE_PHASE) == 0, "flags: only MG_PROT_USE_PHASE is accepted");
    if (const int rc = mg_start_mask(p, start64, start_mask)) return rc;
    return mg_plan_check_prepared(p);
}

static int check_launch(mg_plan *p, int flags, uint64_t start_mask, mg_cds_check *rec, uint32_t *counts, int8_t *junction,
                        cudaStream_t st) {
    mg_genome *g = p->g;
    if (p->n_rec == 0) return MG_OK;
    ChkArgs a;
    a.packed = g->d_packed; a.piece_off = p->d_piece_off; a.piece_src = p->d_piece_src; a.rec_seg_off = p->d_rec_seg_off;
    a.tile_first = p->d_nuc_tile; a.total_dev = p->d_totals; a.cap = p->nuc_total; a.n_rec = p->n_rec; a.stop_mask = p->stop_mask;
    a.rec = rec; a.counts = counts;
    const unsigned rb = (unsigned)((p->n_rec + 255) / 256);
    k_check_records<<<rb, 256, 0, st>>>(a, p->d_rec_phase, (flags & MG_PROT_USE_PHASE) != 0);
    MG_LAUNCH_CHECK();
    if (p->n_nuc_tile > 0) {
        if (counts) k_check_codons<true><<<(unsigned)p->n_nuc_tile, CHK_THREADS, 0, st>>>(a);
        else k_check_codons<false><<<(unsigned)p->n_nuc_tile, CHK_THREADS, 0, st>>>(a);
        MG_LAUNCH_CHECK();
    }
    if (p->n_cseg > 0) {
        k_check_junctions<<<(unsigned)((p->n_cseg + 255) / 256), 256, 0, st>>>(
            p->n_cseg, p->n_rec, p->d_crec_seg_off, p->d_cseg_contig, p->d_cseg_start, p->d_cseg_end, p->d_cseg_strand,
            g->d_contig_len, g->d_contig_base, g->n_contigs, 2 * g->total_bases, g->d_packed, rec, junction);
        MG_LAUNCH_CHECK();
    }
    k_check_final<<<rb, 256, 0, st>>>(p->n_rec, p->stop_mask, start_mask, rec);
    MG_LAUNCH_CHECK();
    return MG_OK;
}

extern "C" int mg_plan_check_device(mg_plan *p, int flags, const uint8_t *start64, mg_cds_check *rec_out, uint32_t *codon_counts,
                                    int8_t *junction, void *stream) {
    uint64_t start_mask = 0;
    if (const int rc = check_args(p, flags, start64, &start_mask)) return rc;
    MG_REQUIRE(p->n_rec == 0 || rec_out != nullptr, "rec_out is NULL");
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    p->last_stream = st;
    return check_launch(p, flags, start_mask, rec_out, codon_counts, junction, st);
}

extern "C" int mg_plan_check(mg_plan *p, int flags, const uint8_t *start64, mg_cds_check *rec_out, uint32_t *codon_counts,
                             int8_t *junction, void *stream) {
    uint64_t start_mask = 0;
    if (const int rc = check_args(p, flags, start64, &start_mask)) return rc;
    MG_REQUIRE(p->n_rec == 0 || rec_out != nullptr, "rec_out is NULL");
    if (p->n_rec == 0) return MG_OK;
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    const bool grow = !p->d_chk || (codon_counts && !p->d_chk_counts) || (junction && p->n_cseg > 0 && !p->d_chk_junction);
    if (grow) {
        if (const int rc = mg_refuse_growth_in_capture(st, "mg_plan_check (first call with these outputs)")) return rc;
        auto alloc = [&](void **d, int64_t bytes) -> int {
            MG_CUDA(cudaMallocAsync(d, std::max<int64_t>(bytes, 1), st));
            p->owned.push_back(*d);
            return MG_OK;
        };
        if (!p->d_chk) if (const int rc = alloc((void **)&p->d_chk, p->n_rec * (int64_t)sizeof(mg_cds_check))) return rc;
        if (codon_counts && !p->d_chk_counts) if (const int rc = alloc((void **)&p->d_chk_counts, p->n_rec * 64 * (int64_t)sizeof(uint32_t))) return rc;
        if (junction && p->n_cseg > 0 && !p->d_chk_junction) if (const int rc = alloc((void **)&p->d_chk_junction, p->n_cseg)) return rc;
    }
    p->last_stream = st;
    int8_t *dj = junction && p->n_cseg > 0 ? p->d_chk_junction : nullptr;
    if (const int rc = check_launch(p, flags, start_mask, p->d_chk, codon_counts ? p->d_chk_counts : nullptr, dj, st)) return rc;
    MG_CUDA(cudaMemcpyAsync(rec_out, p->d_chk, p->n_rec * sizeof(mg_cds_check), cudaMemcpyDeviceToHost, st));
    if (codon_counts)
        MG_CUDA(cudaMemcpyAsync(codon_counts, p->d_chk_counts, p->n_rec * 64 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    if (dj) MG_CUDA(cudaMemcpyAsync(junction, dj, p->n_cseg, cudaMemcpyDeviceToHost, st));
    return MG_OK;
}
