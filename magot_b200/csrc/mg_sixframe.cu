// mg_sixframe.cu -- K4: six-frame translation + stop-codon / ORF scan over whole contigs.
// Replaces Sequence.get_orfs (genome.py:824-851) applied to every contig, i.e. what dna2orfs
// (genome_tools.py:145-180) intended: translations in the order (frame 0,'-'), (0,'+'), (1,'-'),
// (1,'+'), (2,'-'), (2,'+') with the reference's frame quirk (frame 1 == codons from offset 2,
// frame 2 == codons from offset 4, frame 0 == offset 0, or 3 when the first codon is 'X' and is
// trimmed), each split on '*', ORFs shorter than min_aa dropped (min_aa = 0 == reference).
//
// Design: stops are found bit-parallel on the nibble-packed genome (16 positions per 64-bit op, both
// strands from the same forward read: reverse-strand stops TAA/TAG/TGA are TTA/CTA/TCA forward).
// Every stream (contig, frame, strand) is a chain of stops in ascending genome coordinate, bracketed
// by a virtual stop at each contig end; each consecutive pair of stops bounds one ORF, attributed to
// the HIGHER stop.  "Previous stop" is a prefix-max: warp shuffles inside the CTA, a decoupled look-back
// across CTA tiles.  ONE pass over the genome (k_six_scan) finds the stops, counts the kept ORFs per
// (tile, stream) and lists them; a prefix sum of the counts assigns output slots in reference order
// (plus strands ascend, minus strands descend; k_six_place), and the residues are produced by a flat
// 16-residue-per-thread gather like K3 (k_six_aa).  Only when the kept ORFs do not fit the hit list
// (tiny min_aa: an ORF every few bases) a second genome pass writes them (k_six_orfs<true>).
//
// Genetic codes: the stop test is a compile-time expression for the standard code's TAA/TAG/TGA (GEN = false, the default
// kernels) or, for any other code, a loop over the code's stop codons passed as a kernel argument (GEN = true, SixStops).
// The residues come from the call's 4096-entry table.  A code whose stops are the standard three (e.g. table 11) runs the
// default kernels.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include "mg_common.cuh"

#ifndef SIX_THREADS
#define SIX_THREADS 512                              // 24576 bases per CTA: the per-tile prologue (ticket, tile info, look-back) is paid half as often (-12 %)
#endif
#define SIX_HALF 48                                  // bases per stop-mask computation (six_masks)
#ifndef SIX_HALVES
#define SIX_HALVES 3
#endif
#define SIX_BPT (SIX_HALF * SIX_HALVES)              // 144 bases per thread: the per-thread work that does not depend on the number
                                                     // of bases (scans, ranks, ORF tests: about half of the instructions at 48
                                                     // bases per thread) is paid a third as often (measured on config 5:
                                                     // 48 -> 4.77 ms, 96 -> 3.39, 144 -> 2.85, 192 -> 2.94)
#define SIX_FAST_MIN_AA (SIX_BPT / 3)                // two stops of one stream inside a thread are closer than this many codons
#define SIX_TILE (SIX_THREADS * SIX_BPT)             // bases per CTA (multiple of 3 and of 16)
#ifndef SIX_SCAN_MINB
#define SIX_SCAN_MINB 2                             // 64 registers, 32 resident warps per SM (3: 42 registers, 1.2 KB of spill loads per thread, 2.80 vs 2.77 ms)
#endif
#define AA_TILE 8192
#define AA_THREADS 256
#define AA_CAP 512

struct SixHit {                                      // one kept ORF found by the scan pass, placed later (k_six_place)
    int32_t tile, rank;                              // rank among the kept ORFs of (tile, stream), ascending position
    int32_t xl, xh;                                  // contig offsets of the bounding stops
    uint8_t s, xl_real, xh_real, pad;
};

struct mg_sixframe_state {
    int64_t min_aa = 0;
    int32_t *d_cid = nullptr;                        // [nc] the contigs scanned, in output order
    int64_t n_tiles = 0;
    std::vector<int64_t> h_tile_base;                // [n_contig_in_range + 1], starts at 0
    std::vector<int32_t> h_cid;                      // contig ids of the list (kept here so that their upload stays asynchronous)
    int64_t *d_tile_base = nullptr;
    int32_t *d_tile_contig = nullptr;                // [n_tiles] contig (index in the range) of each tile
    int32_t *d_cs = nullptr;                         // [nc*6] first-codon offset of each stream
    int64_t *d_m = nullptr;                          // [nc*6] residues in each stream's translation
    int64_t *d_carry = nullptr;                      // [6][n_tiles] last stop before the tile
    unsigned long long *d_look = nullptr;            // [1 + 6*n_tiles] ticket + look-back status words of the carry max-scan
    struct SixHit *d_hits = nullptr;                 // kept ORFs in discovery order (single-pass path)
    int64_t hit_cap = 0;
    unsigned long long *d_hit_count = nullptr;
    int32_t *d_cnt = nullptr;                        // [n_tiles*6] kept ORFs per (contig, stream, tile) in output order
    int64_t *d_cnt_off = nullptr;                    // [n_tiles*6+1]
    int64_t *d_scan_tmp = nullptr;
    int64_t scan_tmp_cap = 0;
    int64_t n_orf = 0, n_bytes = 0;
    mg_orf *d_recs = nullptr;
    int32_t *d_len = nullptr;
    int64_t *d_aa_off = nullptr;                     // [n_orf+1]
    int64_t *d_src = nullptr;                        // [n_orf] index of the ORF's first base (forward or reverse plane)
    int64_t *d_aa_tile = nullptr;
    int64_t n_aa_tile = 0;
    uint8_t *d_aa = nullptr;                         // library-owned residue buffer for the host variant
    int64_t aa_cap = 0;
    uint8_t *d_aa4096 = nullptr;                     // residue table of a caller's genetic code (NULL: the genome's standard table)
    uint8_t h_aa4096[4096];                          // its host copy (source of the asynchronous upload)
    bool orfcall = false;                            // counted by mg_orfcall_count (records in d_calls) instead of mg_sixframe_count*
    uint64_t generation = 0;                         // g->generation at the count: k_six_aa reads the bases again at emit time
    mg_orfcall *d_calls = nullptr;
    uint8_t *d_start4096 = nullptr;                  // start-codon table of an ORF call (see build_start4096)
    uint8_t h_start4096[4096];
    std::vector<void *> owned;
    bool counted = false;
    bool force_single = false;
    cudaStream_t stream = 0;
};
static thread_local bool g_six_force_single = false;
static int g_six_mode = -1;                          // K4 scan variant (env MAGOT_SIX / mg_tune("six", v)): 0 single pass, 1 two-level on the packed bases, 2 two-level on the stop index (default)
void mg_set_six_mode(int v) { g_six_mode = v; }

// ---- per-stream geometry ------------------------------------------------------------------------------
// stream index sidx = 2*frame + (plus ? 1 : 0): reference order is sidx ascending.
__global__ void k_six_streams(const uint32_t *__restrict__ packed, const int64_t *__restrict__ contig_len,
                              const int64_t *__restrict__ contig_base, const int32_t *__restrict__ cid, int64_t nc,
                              int32_t *__restrict__ cs_out, int64_t *__restrict__ m_out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= nc * 6) return;
    const int64_t c = cid[i / 6];
    const int sidx = (int)(i % 6), f = sidx >> 1, plus = sidx & 1;
    const int64_t L = contig_len[c], gb = contig_base[c];
    int cs = 0;
    int64_t m = 0;
    if (L > 2 + f) {                                 // otherwise translate() returns None (genome.py:810)
        cs = f == 0 ? 0 : (f == 1 ? 2 : 4);
        if (f == 0) {                                // trimX: one leading X is removed (genome.py:819-821)
            const uint64_t v = plus ? mg_ld_nib16(packed, gb) : mg_ld_nib16(packed, gb + L - 3);
            if ((uint32_t)v & 0x888u) cs = 3;        // complementing does not change validity
        }
        m = (L - cs) / 3;
        if (m < 0) m = 0;
    }
    cs_out[i] = cs;
    m_out[i] = m;
}

// The same for ORF calling: true phases, no trimX.  Stream sidx reads residue class stream_res(sidx), so frame f = sidx >> 1
// is phase 0, 2, 1 for f = 0, 1, 2 (the quirk's offsets 0, 2, 4 modulo 3).
__global__ void k_orf_streams(const int64_t *__restrict__ contig_len, const int32_t *__restrict__ cid, int64_t nc,
                              int32_t *__restrict__ cs_out, int64_t *__restrict__ m_out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= nc * 6) return;
    const int f = (int)(i % 6) >> 1, phase = f == 0 ? 0 : (f == 1 ? 2 : 1);
    const int64_t L = contig_len[cid[i / 6]];
    cs_out[i] = phase;
    m_out[i] = L > phase ? (L - phase) / 3 : 0;
}

// ---- stop masks of one thread's 48 positions ---------------------------------------------------------
#define NIBM 0x1111111111111111ull
__device__ __forceinline__ uint64_t res_mask(int r) {     // nibble slots k with k % 3 == r
    return r == 0 ? 0x1001001001001001ull : (r == 1 ? 0x0010010010010010ull : 0x0100100100100100ull);
}

struct SixMasks {
    uint64_t pm[3], mm[3];                           // plus / minus stop flags, bit 4k of group g = position 16g+k
};

// Stop codons of a non-standard genetic code, codon index 16*b0 + 4*b1 + b2 (A=0 C=1 G=2 T=3).  Passed by value as a
// __grid_constant__ kernel argument: the loop over the codons reads the constant bank.
struct SixStops {
    int32_t n;                                       // 0..64
    uint8_t fwd[64];                                 // the stops, read on the plus strand
    uint8_t rev[64];                                 // their reverse complements: the minus-strand stops as read forward
};
#define SIX_STD_STOPS ((1ull << 48) | (1ull << 50) | (1ull << 56))   // TAA TAG TGA: the stop set of the GEN = false kernels

__device__ __forceinline__ uint64_t pick_plane(int b, uint64_t a, uint64_t c, uint64_t g, uint64_t t) {
    return (b & 2) ? ((b & 1) ? t : g) : ((b & 1) ? c : a);
}

// x0 = contig offset of the thread's first position (multiple of 48); gb = contig's global base index
// WHICH: 0 = both strands, 1 = plus only (s.mm undefined), 2 = minus only (s.pm undefined)
// GEN: stops from `ss` instead of TAA/TAG/TGA (ss is not read when GEN is false)
template <int WHICH, bool GEN>
__device__ __forceinline__ void six_masks_t(const uint32_t *__restrict__ packed, int64_t gb, int64_t L, int64_t x0,
                                            const int32_t *cs6, const SixStops &ss, SixMasks &s) {
    uint64_t v[4];
    const uint2 *p = reinterpret_cast<const uint2 *>(packed + ((gb + x0) >> 3));
#pragma unroll
    for (int g = 0; g < 3; g++) {
        const uint2 w = __ldg(p + g);
        v[g] = ((uint64_t)w.y << 32) | w.x;
    }
    v[3] = __ldg(packed + ((gb + x0 + 48) >> 3));   // only nibbles 48,49 are needed
    uint64_t T[4], A[4], G[4], C[4];
#pragma unroll
    for (int g = 0; g < 4; g++) {
        const uint64_t inv = (v[g] >> 3) & NIBM, b0 = v[g] & NIBM, b1 = (v[g] >> 1) & NIBM;
        T[g] = b1 & b0 & ~inv;
        A[g] = NIBM & ~(b1 | b0 | inv);
        G[g] = b1 & ~b0 & ~inv;
        C[g] = b0 & ~b1 & ~inv;
    }
#pragma unroll
    for (int g = 0; g < 3; g++) {
        const uint64_t A1 = (A[g] >> 4) | (A[g + 1] << 60), A2 = (A[g] >> 8) | (A[g + 1] << 56);
        const uint64_t G1 = (G[g] >> 4) | (G[g + 1] << 60), G2 = (G[g] >> 8) | (G[g + 1] << 56);
        const uint64_t T1 = (T[g] >> 4) | (T[g + 1] << 60);
        const uint64_t C1 = (C[g] >> 4) | (C[g + 1] << 60);
        if (!GEN) {
            if (WHICH != 2) s.pm[g] = T[g] & ((A1 & (A2 | G2)) | (G1 & A2));          // TAA TAG TGA
            if (WHICH != 1) s.mm[g] = A2 & ((T1 & (T[g] | C[g])) | (C1 & T[g]));      // TTA CTA TCA = rc of the above
        } else {
            // every stop codon b0 b1 b2: the AND of the planes of b0, b1, b2 at offsets 0, 1, 2
            const uint64_t T2 = (T[g] >> 8) | (T[g + 1] << 56), C2 = (C[g] >> 8) | (C[g + 1] << 56);
            uint64_t pm = 0, mm = 0;
#pragma unroll 1
            for (int i = 0; i < ss.n; i++) {
                if (WHICH != 2) {
                    const int c = ss.fwd[i];
                    pm |= pick_plane(c >> 4, A[g], C[g], G[g], T[g]) & pick_plane((c >> 2) & 3, A1, C1, G1, T1) &
                          pick_plane(c & 3, A2, C2, G2, T2);
                }
                if (WHICH != 1) {
                    const int c = ss.rev[i];
                    mm |= pick_plane(c >> 4, A[g], C[g], G[g], T[g]) & pick_plane((c >> 2) & 3, A1, C1, G1, T1) &
                          pick_plane(c & 3, A2, C2, G2, T2);
                }
            }
            if (WHICH != 2) s.pm[g] = pm;
            if (WHICH != 1) s.mm[g] = mm;
        }
    }
    // ---- validity at the contig ends
    const int64_t lim = L - 2 - x0;                  // positions t >= lim have no full codon
    if (lim < 48) {
#pragma unroll
        for (int g = 0; g < 3; g++) {
            const int64_t k = lim - 16 * g;
            const uint64_t keep = k <= 0 ? 0ull : (k >= 16 ? ~0ull : ((1ull << (4 * k)) - 1ull));
            if (WHICH != 2) s.pm[g] &= keep;
            if (WHICH != 1) s.mm[g] &= keep;
        }
    }
    if (WHICH != 2 && x0 == 0) {
        if (cs6[1] == 3) s.pm[0] &= ~1ull;           // frame 0 '+': trimmed first codon
        s.pm[0] &= ~(1ull << 4);                     // frame 2 '+' starts at offset 4: codon at 1 is not read
    }
    // minus strand: oriented start q0 = L-3-x; frame 0 trimmed drops q0 = 0, frame 2 never reads q0 = 1
    if (WHICH != 1) {
        const int64_t t0 = L - 3 - x0, t1 = L - 4 - x0;
        if (cs6[0] == 3 && t0 >= 0 && t0 < 48) s.mm[t0 >> 4] &= ~(1ull << (4 * (t0 & 15)));
        if (t1 >= 0 && t1 < 48) s.mm[t1 >> 4] &= ~(1ull << (4 * (t1 & 15)));
    }
}

template <bool GEN>
__device__ __forceinline__ void six_masks(const uint32_t *__restrict__ packed, int64_t gb, int64_t L, int64_t x0,
                                          const int32_t *cs6, const SixStops &ss, SixMasks &s) {
    six_masks_t<0, GEN>(packed, gb, L, x0, cs6, ss, s);
}

// residue (t % 3) selected by stream sidx: plus frame f -> rho_f, minus -> (L%3 - rho_f) % 3
__device__ __forceinline__ int stream_res(int sidx, int Lm3) {
    const int f = sidx >> 1;
    const int rho = f == 0 ? 0 : (f == 1 ? 2 : 1);
    return (sidx & 1) ? rho : (Lm3 - rho + 3) % 3;
}

// ---- position-ordered stop masks --------------------------------------------------------------------------------------
// The nibble-spaced flags of one strand (3 x 64 bits) are compressed to one bit per position (48 bits): first / last stop
// of a stream are then one masked ffs / clz per half instead of three per stream on nibble-spaced words (that extraction
// was 29 % of the scan kernel's instructions), and walking the stops of a stream is a plain bit loop.
__device__ __forceinline__ uint32_t compress8(uint32_t x) {       // flags at bits 0, 4, .., 28 -> bits 0..7
    x = (x | (x >> 3)) & 0x03030303u;
    x = (x | (x >> 6)) & 0x000F000Fu;
    return (x | (x >> 12)) & 0xFFu;
}
__device__ __forceinline__ uint64_t pos48(const uint64_t m[3]) {
    const uint32_t lo = compress8((uint32_t)m[0]) | (compress8((uint32_t)(m[0] >> 32)) << 8) | (compress8((uint32_t)m[1]) << 16) |
                        (compress8((uint32_t)(m[1] >> 32)) << 24);
    const uint32_t hi = compress8((uint32_t)m[2]) | (compress8((uint32_t)(m[2] >> 32)) << 8);
    return ((uint64_t)hi << 32) | lo;
}
// stops of one thread's SIX_BPT positions, one bit per position: half h covers positions 48h .. 48h+47
struct ThreadStops {
    uint64_t p[SIX_HALVES], m[SIX_HALVES];           // plus / minus strand
};
// the stops of stream sidx (a residue class of one strand).  Both halves start at a multiple of 3, so one residue mask serves.
__device__ __forceinline__ void stream_stops(const ThreadStops &ts, int sidx, int Lm3, uint64_t x[SIX_HALVES]) {
    const uint64_t rm = 0x0000249249249249ull << stream_res(sidx, Lm3);
#pragma unroll
    for (int h = 0; h < SIX_HALVES; h++) x[h] = ((sidx & 1) ? ts.p[h] : ts.m[h]) & rm;
}
__device__ __forceinline__ void stops_first_last(const uint64_t x[SIX_HALVES], int &first, int &last) {
    // selects, not branches: the halves that hold a stop differ from lane to lane (as branches these lines were 17 % of
    // the scan's instructions at 12-20 active lanes)
    first = -1;
    last = -1;
#pragma unroll
    for (int h = SIX_HALVES - 1; h >= 0; h--) {
        const int f = __ffsll((long long)x[h]);      // 0 when the half holds no stop
        first = f ? SIX_HALF * h + f - 1 : first;
    }
#pragma unroll
    for (int h = 0; h < SIX_HALVES; h++) {
        const int l = SIX_HALF * h + 63 - __clzll((long long)x[h]);
        last = x[h] ? l : last;
    }
}

struct TileInfo;

struct TileInfo {
    int64_t c, ci, k, gb, L, Tc;                     // contig, its index in the scanned list, tile index in contig, global base, length, tiles in contig
    int64_t vb;                                      // scan coordinate of the contig's first base: tile_base[ci] * SIX_TILE.  Stops are
                                                     // carried between tiles in this coordinate (it ascends with the tile index
                                                     // whatever the order of the contig list; a genome index would not)
    int Lm3;
    int32_t cs[6];
    int64_t m[6];
};

// thread per tile: index (within the scanned range) of the contig that owns the tile
__global__ void __launch_bounds__(256) k_six_tile_contig(const int64_t *__restrict__ tile_base, int64_t nc, int64_t n_tiles,
                                                         int32_t *__restrict__ tile_contig) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    int64_t lo = 0, hi = nc;                          // largest ci with tile_base[ci] <= t (contigs without tiles: the last one)
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (tile_base[mid] <= t) lo = mid; else hi = mid;
    }
    tile_contig[t] = (int32_t)lo;
}

// tile_info with the contig index already known (k_six_tile_contig): independent loads, no search
__device__ __forceinline__ void tile_info_at(int64_t tile, int64_t lo, const int64_t *__restrict__ tile_base, const int32_t *__restrict__ cid,
                                             const int64_t *__restrict__ contig_len, const int64_t *__restrict__ contig_base,
                                             const int32_t *__restrict__ cs, const int64_t *__restrict__ m, struct TileInfo &ti);

__device__ __forceinline__ void tile_info(int64_t tile, const int64_t *__restrict__ tile_base, int64_t nc, const int32_t *__restrict__ cid,
                                          const int64_t *__restrict__ contig_len, const int64_t *__restrict__ contig_base,
                                          const int32_t *__restrict__ cs, const int64_t *__restrict__ m, TileInfo &ti) {
    int64_t lo = 0, hi = nc;                          // largest ci with tile_base[ci] <= tile
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (tile_base[mid] <= tile) lo = mid; else hi = mid;
    }
    // contigs without tiles (L == 0) share a tile_base value with their successor: take the last one
    ti.c = cid[lo];
    ti.ci = lo;
    ti.k = tile - tile_base[lo];
    ti.Tc = tile_base[lo + 1] - tile_base[lo];
    ti.gb = contig_base[ti.c];
    ti.vb = tile_base[lo] * SIX_TILE;
    ti.L = contig_len[ti.c];
    ti.Lm3 = (int)(ti.L % 3);
#pragma unroll
    for (int s = 0; s < 6; s++) {
        ti.cs[s] = cs[lo * 6 + s];
        ti.m[s] = m[lo * 6 + s];
    }
}

__device__ __forceinline__ void tile_info_at(int64_t tile, int64_t lo, const int64_t *__restrict__ tile_base, const int32_t *__restrict__ cid,
                                             const int64_t *__restrict__ contig_len, const int64_t *__restrict__ contig_base,
                                             const int32_t *__restrict__ cs, const int64_t *__restrict__ m, TileInfo &ti) {
    ti.c = cid[lo];
    ti.ci = lo;
    ti.k = tile - tile_base[lo];
    ti.Tc = tile_base[lo + 1] - tile_base[lo];
    ti.gb = contig_base[ti.c];
    ti.vb = tile_base[lo] * SIX_TILE;
    ti.L = contig_len[ti.c];
    ti.Lm3 = (int)(ti.L % 3);
#pragma unroll
    for (int s = 0; s < 6; s++) {
        ti.cs[s] = cs[lo * 6 + s];
        ti.m[s] = m[lo * 6 + s];
    }
}

template <bool GEN>
__device__ __forceinline__ void thread_stops(const uint32_t *__restrict__ packed, const TileInfo &ti, int64_t x0, const SixStops &ss,
                                             ThreadStops &ts) {
#pragma unroll
    for (int h = 0; h < SIX_HALVES; h++) {
        const int64_t xh = x0 + SIX_HALF * h;
        if (xh < ti.L) {
            SixMasks sm;
            six_masks<GEN>(packed, ti.gb, ti.L, xh, ti.cs, ss, sm);
            ts.p[h] = pos48(sm.pm);
            ts.m[h] = pos48(sm.mm);
        } else {
            ts.p[h] = 0;
            ts.m[h] = 0;
        }
    }
}

// ---- ORF enumeration shared by the single-pass scan (k_six_scan) and the dense-output second pass (k_six_orfs) ----
// ORF between a lower stop xl and a higher stop xh of one stream (contig offsets; !xl_real = virtual stop at
// the low end of the contig, !xh_real = virtual stop at the high end).  Residue index of a stop at x:
// plus (x-cs)/3, minus (L-3-cs-x)/3 (descending in x).
__device__ __forceinline__ void orf_of(int plus, int64_t L, int cs, int64_t m, int64_t xl, int64_t xh, bool xl_real,
                                       bool xh_real, int64_t &start, int64_t &len) {
    if (plus) {
        const int64_t il = xl_real ? (xl - cs) / 3 : -1;
        const int64_t ih = xh_real ? (xh - cs) / 3 : m;
        start = il + 1;
        len = ih - il - 1;
    } else {
        const int64_t il = xl_real ? (L - 3 - cs - xl) / 3 : m;
        const int64_t ih = xh_real ? (L - 3 - cs - xh) / 3 : -1;
        start = ih + 1;
        len = il - ih - 1;
    }
}

__device__ __forceinline__ int64_t layout_index(const TileInfo &ti, const int64_t *__restrict__ tile_base, int s) {
    // output order: contig, then stream (reference order), then tiles ascending ('+') or descending ('-')
    return tile_base[ti.ci] * 6 + (int64_t)s * ti.Tc + ((s & 1) ? ti.k : ti.Tc - 1 - ti.k);
}

// Enumerate the ORFs this thread owns in stream s (each ORF belongs to its higher stop).  WRITE == false: count.
// WRITE == true: k-th kept ORF (ascending position) goes to slot0 + k ('+') or slot0 + (n_mine-1-k) ('-').
// WRITE == 2: k-th kept ORF goes to hits[slot0 + k] with rank n_mine + k (n_mine = kept ORFs of lower threads).
template <int WRITE>
__device__ __forceinline__ int enumerate_stream(const TileInfo &ti, const ThreadStops &ts, int s, int64_t x0, int64_t prev,
                                                bool is_end_thread, int64_t min_aa, int64_t two_T, int64_t slot0, int n_mine,
                                                mg_orf *__restrict__ recs, int32_t *__restrict__ lens, int64_t *__restrict__ srcs,
                                                SixHit *__restrict__ hits = nullptr, int32_t tile = 0, int fl = -2) {
    if (ti.m[s] <= 0) return 0;                       // `if translated_seq:` (genome.py:832)
    const int plus = s & 1;
    int k = 0;
    // one candidate ORF: between stops xl (lower) and xh (higher, !real = virtual stop at the contig's high end)
    // Contig offsets fit 32 bits (mg_sixframe_count rejects longer contigs).  The length test needs no division:
    // both stops are congruent to cs modulo 3, so len = span/3 - 1; the divisions of orf_of run for kept ORFs only.
    const int32_t L32 = (int32_t)ti.L, cs32 = ti.cs[s], m32 = (int32_t)ti.m[s];
    const int64_t need3 = 3 * min_aa;                       // residues * 3
    auto visit = [&](int64_t xl, bool xl_real, int64_t xh, bool real) {
        // span3 = 3 * (number of residues of the candidate)
        const int32_t ql = plus ? (int32_t)xl - cs32 : L32 - 3 - cs32 - (int32_t)xl;   // 3 * residue index of the lower stop
        const int32_t qh = plus ? (int32_t)xh - cs32 : L32 - 3 - cs32 - (int32_t)xh;
        int64_t span3;
        if (plus) span3 = (int64_t)(real ? qh : 3 * m32) - (xl_real ? ql : -3) - 3;
        else span3 = (int64_t)(xl_real ? ql : 3 * m32) - (real ? qh : -3) - 3;
        if (span3 >= need3) {
            if (WRITE == 2) {
                SixHit h;
                h.tile = tile; h.rank = n_mine + k; h.xl = (int32_t)xl; h.xh = (int32_t)xh;
                h.s = (uint8_t)s; h.xl_real = xl_real; h.xh_real = real; h.pad = 0;
                hits[slot0 + k] = h;
            } else if (WRITE == 1) {
                int64_t st, ln;
                orf_of(plus, ti.L, ti.cs[s], ti.m[s], xl, xh, xl_real, real, st, ln);
                const int64_t slot = slot0 + (plus ? k : n_mine - 1 - k);
                mg_orf o;
                o.contig = (int32_t)ti.c; o.frame = (int8_t)(s >> 1); o.minus = (int8_t)(!plus); o.pad = 0;
                o.start = st; o.len = ln; o.aa_off = 0;
                recs[slot] = o;
                lens[slot] = (int32_t)ln;
                const int64_t q = ti.cs[s] + 3 * st;                // oriented offset of the ORF's first base
                srcs[slot] = plus ? (ti.gb + q) : (two_T - ti.gb - ti.L + q);      // '-': forward read of the reverse plane
            }
            k++;
        }
    };
    uint64_t x[SIX_HALVES];
    if (min_aa >= SIX_FAST_MIN_AA) {
        // Two stops of one stream inside a thread's SIX_BPT bases are < SIX_BPT/3 codons apart, so only the FIRST stop of the
        // thread (and the virtual stop at the contig end) can close an ORF of that many residues: no loop over stops.
        int first, last;                              // fl: (first, last) packed by the caller, -2 = not known
        if (fl != -2) { first = (fl & 0xFF) - 1; last = ((fl >> 8) & 0xFF) - 1; }
        else { stream_stops(ts, s, ti.Lm3, x); stops_first_last(x, first, last); }
        if (first >= 0) visit(prev, prev >= 0, x0 + first, true);
        if (is_end_thread) {
            const int64_t xl = last >= 0 ? x0 + last : prev;
            visit(xl, xl >= 0, 0, false);
        }
        return k;
    }
    stream_stops(ts, s, ti.Lm3, x);
    int64_t xl = prev;
    bool xl_real = prev >= 0;
#pragma unroll
    for (int h = 0; h < SIX_HALVES; h++) {
        uint64_t v = x[h];
        while (v) {
            const int64_t xh = x0 + SIX_HALF * h + __ffsll((long long)v) - 1;
            v &= v - 1;
            visit(xl, xl_real, xh, true);
            xl = xh;
            xl_real = true;
        }
    }
    if (is_end_thread) visit(xl, xl_real, 0, false);  // the virtual stop at the contig's high end
    return k;
}

__device__ __forceinline__ int64_t warp_incl_sum(int64_t v) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += t;
    }
    return v;
}
__device__ __forceinline__ int64_t block_incl_sum(int64_t v, int64_t *s_warp, int64_t *total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    v = warp_incl_sum(v);
    if (lane == 31) s_warp[wid] = v;
    __syncthreads();
    if (wid == 0) {
        int64_t w = lane < (SIX_THREADS / 32) ? s_warp[lane] : 0;
        w = warp_incl_sum(w);
        if (lane < (SIX_THREADS / 32)) s_warp[lane] = w;
    }
    __syncthreads();
    const int64_t off = wid ? s_warp[wid - 1] : 0;
    *total = s_warp[SIX_THREADS / 32 - 1];
    __syncthreads();
    return v + off;
}

template <bool EMIT, bool GEN>
__global__ void __launch_bounds__(SIX_THREADS) k_six_orfs(
    const uint32_t *__restrict__ packed, const int64_t *__restrict__ tile_base, int64_t nc, const int32_t *__restrict__ cid,
    const int64_t *__restrict__ contig_len, const int64_t *__restrict__ contig_base, const int32_t *__restrict__ cs,
    const int64_t *__restrict__ m, int64_t n_tiles, const int64_t *__restrict__ carry, int64_t min_aa, int64_t two_T,
    int32_t *__restrict__ cnt, const int64_t *__restrict__ cnt_off, mg_orf *__restrict__ recs, int32_t *__restrict__ lens,
    int64_t *__restrict__ srcs, const __grid_constant__ SixStops ss) {
    __shared__ TileInfo ti;
    __shared__ int s_cnt[6];
    __shared__ int64_t s_warp[SIX_THREADS / 32];
    __shared__ int s_wlast[6][SIX_THREADS / 32];     // per-warp max of `last stop in thread`
    if (threadIdx.x == 0) tile_info(blockIdx.x, tile_base, nc, cid, contig_len, contig_base, cs, m, ti);
    if (threadIdx.x < 6) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const int64_t tile0 = ti.k * SIX_TILE;
    const int64_t x0 = tile0 + (int64_t)threadIdx.x * SIX_BPT;
    const bool active = x0 < ti.L;
    const bool is_end_thread = active && (x0 + SIX_BPT >= ti.L);       // owns the virtual high-end stops
    ThreadStops sm;                                   // the thread's stops, one bit per position
    if (active) thread_stops<GEN>(packed, ti, x0, ss, sm);
    else { for (int h = 0; h < SIX_HALVES; h++) { sm.p[h] = 0; sm.m[h] = 0; } }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;

    // previous stop of each stream before this thread: exclusive max over lower threads, else the tile carry
    int ex_local[6];
#pragma unroll
    for (int s = 0; s < 6; s++) {
        int first, last;
        uint64_t xs[SIX_HALVES];
        stream_stops(sm, s, ti.Lm3, xs);
        stops_first_last(xs, first, last);
        int inc = last < 0 ? -1 : (int)threadIdx.x * SIX_BPT + last;   // tile-local position
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d && t > inc) inc = t;
        }
        if (lane == 31) s_wlast[s][wid] = inc;
        int ex = __shfl_up_sync(0xffffffffu, inc, 1);
        if (lane == 0) ex = -1;
        ex_local[s] = ex;
    }
    __syncthreads();
    int64_t prev[6];
#pragma unroll
    for (int s = 0; s < 6; s++) {
        int ex = ex_local[s];
        for (int w = 0; w < wid; w++) ex = max(ex, s_wlast[s][w]);
        if (ex >= 0) prev[s] = tile0 + ex;            // contig offset
        else {
            const int64_t cg = carry[(int64_t)s * n_tiles + blockIdx.x];   // scan coordinate; < vb: other contig
            prev[s] = (cg >= ti.vb) ? cg - ti.vb : -1;
        }
    }

    int my_cnt[6];
#pragma unroll
    for (int s = 0; s < 6; s++)
        my_cnt[s] = active ? enumerate_stream<0>(ti, sm, s, x0, prev[s], is_end_thread, min_aa, two_T, 0, 0, nullptr, nullptr, nullptr) : 0;

    if (!EMIT) {
#pragma unroll
        for (int s = 0; s < 6; s++) {
            int c = my_cnt[s];
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
            if (lane == 0 && c) atomicAdd(&s_cnt[s], c);
        }
        __syncthreads();
        if (threadIdx.x < 6) cnt[layout_index(ti, tile_base, threadIdx.x)] = s_cnt[threadIdx.x];
    } else {
        // ranks inside the tile: block prefix sums of the per-thread counts, three 21-bit fields per word
        const int64_t pk0 = (int64_t)my_cnt[0] | ((int64_t)my_cnt[1] << 21) | ((int64_t)my_cnt[2] << 42);
        const int64_t pk1 = (int64_t)my_cnt[3] | ((int64_t)my_cnt[4] << 21) | ((int64_t)my_cnt[5] << 42);
        int64_t tot0, tot1;
        const int64_t in0 = block_incl_sum(pk0, s_warp, &tot0);
        const int64_t in1 = block_incl_sum(pk1, s_warp, &tot1);
        if (active) {
#pragma unroll
            for (int s = 0; s < 6; s++) {
                if (my_cnt[s] == 0) continue;
                const int sh = 21 * (s % 3);
                const int64_t inc = ((s < 3 ? in0 : in1) >> sh) & 0x1FFFFF;
                const int64_t tot = ((s < 3 ? tot0 : tot1) >> sh) & 0x1FFFFF;
                // '+': ascending, my first ORF has rank = exclusive prefix; '-': descending, ranks count from the top
                const int64_t rank0 = (s & 1) ? inc - my_cnt[s] : tot - inc;
                const int64_t slot0 = cnt_off[layout_index(ti, tile_base, s)] + rank0;
                enumerate_stream<1>(ti, sm, s, x0, prev[s], is_end_thread, min_aa, two_T, slot0, my_cnt[s], recs, lens, srcs);
            }
        }
    }
}

// ---- single pass: stops, carry, count and the kept ORFs themselves ------------------------------------------------
// Replaces pass A (k_six_last), pass B (k_ms_*) and pass C (k_six_orfs<false>), and -- when the kept ORFs fit the hit
// buffer, which they do for any practical min_aa -- pass D (k_six_orfs<true>) as well: the genome is read ONCE.
//  * the carry (last stop of each stream before the tile) comes from a decoupled look-back over the tiles' own last
//    stops.  Stop positions ascend with the tile index, so a tile that contains a stop publishes its inclusive prefix at
//    once and the look-back of its successor ends after one step; warps 0..5 do the six streams in parallel.
//  * kept ORFs are rare (one per ~3 kb for min_aa = 100): they are appended to a hit list in discovery order (one atomic
//    per tile) with their rank inside (tile, stream); k_six_place puts them into reference order after the prefix sum of
//    the per-(tile, stream) counts.
#define SIX_LOOK_NONE 0ull
#define SIX_LOOK_SUM (1ull << 62)                    // tile has no stop in this stream, prefix not known yet
#define SIX_LOOK_PREFIX (2ull << 62)                 // value = 1 + last stop at or before the end of this tile (0 = none)
#define SIX_LOOK_MASK (3ull << 62)

template <bool GEN>
__global__ void __launch_bounds__(SIX_THREADS, SIX_SCAN_MINB) k_six_scan(
    const uint32_t *__restrict__ packed, const int64_t *__restrict__ tile_base, int64_t nc, const int32_t *__restrict__ cid,
    const int64_t *__restrict__ contig_len, const int64_t *__restrict__ contig_base, const int32_t *__restrict__ cs,
    const int64_t *__restrict__ m, const int32_t *__restrict__ tile_contig, int64_t n_tiles, unsigned long long *look, int64_t *__restrict__ carry_out, int64_t min_aa,
    int64_t two_T, int32_t *__restrict__ cnt, SixHit *__restrict__ hits, int64_t hit_cap, unsigned long long *hit_count,
    const __grid_constant__ SixStops ss) {
    __shared__ TileInfo ti;
    __shared__ int64_t s_warp[SIX_THREADS / 32];
    __shared__ int s_wlast[6][SIX_THREADS / 32];     // per-warp max of `last stop in thread`
    __shared__ int64_t s_carry[6];                   // last stop of each stream before the tile (contig offset, -1 = none)
    __shared__ int64_t s_tile;
    __shared__ long long s_base;
    if (threadIdx.x == 0) {
        const int64_t t = (int64_t)atomicAdd(look, 1ull);              // tiles in launch order: look-back never waits on a
        s_tile = t;                                                      // tile that has not started
        tile_info_at(t, tile_contig[t], tile_base, cid, contig_len, contig_base, cs, m, ti);
    }
    __syncthreads();
    const int64_t tile = s_tile;
    const int64_t tile0 = ti.k * SIX_TILE;
    const int64_t x0 = tile0 + (int64_t)threadIdx.x * SIX_BPT;
    const bool active = x0 < ti.L;
    const bool is_end_thread = active && (x0 + SIX_BPT >= ti.L);       // owns the virtual high-end stops
    ThreadStops sm;                                   // the thread's stops, one bit per position
    if (active) thread_stops<GEN>(packed, ti, x0, ss, sm);
    else { for (int h = 0; h < SIX_HALVES; h++) { sm.p[h] = 0; sm.m[h] = 0; } }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;

    int ex_local[6], fl[6];                          // fl: (first + 1) | (last + 1) << 8 of the thread's stops per stream
#pragma unroll
    for (int s = 0; s < 6; s++) {
        int first, last;
        uint64_t xs[SIX_HALVES];
        stream_stops(sm, s, ti.Lm3, xs);
        stops_first_last(xs, first, last);
        fl[s] = (first + 1) | ((last + 1) << 8);
        int inc = last < 0 ? -1 : (int)threadIdx.x * SIX_BPT + last;   // tile-local position
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d && t > inc) inc = t;
        }
        if (lane == 31) s_wlast[s][wid] = inc;
        int ex = __shfl_up_sync(0xffffffffu, inc, 1);
        if (lane == 0) ex = -1;
        ex_local[s] = ex;
    }
    __syncthreads();
    // Every warp: last stop of each stream in the warps before it (one 16-lane max-scan per stream, no barrier), so that only
    // the few threads in front of a stream's first stop in the tile depend on the carry from earlier tiles.
    constexpr int NW = SIX_THREADS / 32;
    int64_t prev[6];                                  // contig offset of the last stop of the stream before this thread, -1 = none
    unsigned int need = 0;                            // streams whose prev is the carry (not known yet)
    int my_agg = -1;                                  // warp s < 6: the tile's last stop of stream s
#pragma unroll
    for (int s = 0; s < 6; s++) {
        int inc = lane < NW ? s_wlast[s][lane] : -1;
#pragma unroll
        for (int d = 1; d < NW; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d && t > inc) inc = t;
        }
        const int exw = __shfl_sync(0xffffffffu, inc, wid ? wid - 1 : 0);
        const int agg = __shfl_sync(0xffffffffu, inc, NW - 1);
        if (s == wid) my_agg = agg;
        if (ex_local[s] >= 0) prev[s] = tile0 + ex_local[s];
        else if (wid && exw >= 0) prev[s] = tile0 + exw;
        else { prev[s] = -1; need |= 1u << s; }
    }
    // publish the tile's own last stops at once: the successor's look-back finds them while this tile is still counting
    if (wid < 6 && lane == 0) {
        volatile unsigned long long *st = look + 1 + (int64_t)wid * n_tiles;
        const unsigned long long own = my_agg >= 0 ? (unsigned long long)(ti.vb + tile0 + my_agg + 1) : 0ull;
        st[tile] = (my_agg >= 0 || tile == 0) ? (SIX_LOOK_PREFIX | own) : SIX_LOOK_SUM;
    }
    int my_cnt[6];
    int mine = 0;
#pragma unroll
    for (int s = 0; s < 6; s++) {
        my_cnt[s] = (active && !((need >> s) & 1u))
                        ? enumerate_stream<0>(ti, sm, s, x0, prev[s], is_end_thread, min_aa, two_T, 0, 0, nullptr, nullptr, nullptr, nullptr, 0, fl[s])
                        : 0;
        mine += my_cnt[s];
    }
    if (wid < 6) {                                    // warp s: look back for the carry of stream s (by now usually published)
        const int s = wid;
        volatile unsigned long long *st = look + 1 + (int64_t)s * n_tiles;
        unsigned long long best = 0;                  // 1 + last stop before this tile, 0 = none
        int64_t j = tile - 1 - lane;
        while (true) {
            unsigned long long w = SIX_LOOK_PREFIX;   // before tile 0: nothing
            if (j >= 0) { while (((w = st[j]) & SIX_LOOK_MASK) == SIX_LOOK_NONE) __nanosleep(64); }
            const unsigned int done = __ballot_sync(0xffffffffu, (w & SIX_LOOK_MASK) == SIX_LOOK_PREFIX);
            if (done) {                               // nearest tile with a known prefix; tiles nearer than it hold no stop
                best = __shfl_sync(0xffffffffu, w & ~SIX_LOOK_MASK, __ffs(done) - 1);
                break;
            }
            j -= 32;
        }
        const int64_t cg = (int64_t)best - 1;         // scan coordinate; < vb: a stop of another contig
        if (lane == 0) {
            s_carry[s] = cg >= ti.vb ? cg - ti.vb : -1;
            carry_out[(int64_t)s * n_tiles + tile] = cg;
            if (my_agg < 0 && tile > 0) st[tile] = SIX_LOOK_PREFIX | best;
        }
    }
    __syncthreads();
    if (need && active) {                             // the threads in front of the first stop of a stream
#pragma unroll
        for (int s = 0; s < 6; s++) {
            if (!((need >> s) & 1u)) continue;
            prev[s] = s_carry[s];
            my_cnt[s] = enumerate_stream<0>(ti, sm, s, x0, prev[s], is_end_thread, min_aa, two_T, 0, 0, nullptr, nullptr, nullptr, nullptr, 0, fl[s]);
            mine += my_cnt[s];
        }
    }
    int tot[6], before[6], excl[6];                   // kept ORFs of the tile per stream; of the streams before s; of lower threads
    int run = 0;
    if (min_aa >= SIX_FAST_MIN_AA) {
        // a thread keeps at most two ORFs per stream (its first stop, the contig end): ranks from two ballots per stream and
        // the per-warp totals, one barrier; only the rare threads that hold an ORF read the totals back
        __shared__ int s_wcnt[6][NW];
        const unsigned int lt = (1u << lane) - 1u;
        int ex_w[6];
#pragma unroll
        for (int s = 0; s < 6; s++) {
            const unsigned int b1 = __ballot_sync(0xffffffffu, my_cnt[s] >= 1), b2 = __ballot_sync(0xffffffffu, my_cnt[s] >= 2);
            ex_w[s] = __popc(b1 & lt) + __popc(b2 & lt);
            if (lane == 0) s_wcnt[s][wid] = __popc(b1) + __popc(b2);
        }
        __syncthreads();
        if (threadIdx.x < 6) {
            int t = 0;
#pragma unroll
            for (int w = 0; w < NW; w++) t += s_wcnt[threadIdx.x][w];
            cnt[layout_index(ti, tile_base, threadIdx.x)] = t;
        }
        if (mine == 0) return;
        // every holder claims room in the hit list for its own ORFs (their order in the list does not matter)
        const long long base = (long long)atomicAdd(hit_count, (unsigned long long)mine);
        if (base + mine > hit_cap) return;            // overflow: the host falls back to the two-pass emit
        int off = 0;
#pragma unroll
        for (int s = 0; s < 6; s++) {
            if (my_cnt[s] == 0) continue;
            int e = ex_w[s];                          // kept ORFs of the stream in lower threads of the tile
            for (int w = 0; w < wid; w++) e += s_wcnt[s][w];
            enumerate_stream<2>(ti, sm, s, x0, prev[s], is_end_thread, min_aa, two_T, base + off, e, nullptr, nullptr, nullptr,
                                hits, (int32_t)tile, fl[s]);
            off += my_cnt[s];
        }
        return;
    }
    const int any = __syncthreads_or(mine);
    if (!any) {
        if (threadIdx.x < 6) cnt[layout_index(ti, tile_base, threadIdx.x)] = 0;
        return;
    }
    // general case: block prefix sums of the per-thread counts, three 21-bit fields per word
    const int64_t pk0 = (int64_t)my_cnt[0] | ((int64_t)my_cnt[1] << 21) | ((int64_t)my_cnt[2] << 42);
    const int64_t pk1 = (int64_t)my_cnt[3] | ((int64_t)my_cnt[4] << 21) | ((int64_t)my_cnt[5] << 42);
    int64_t tot0, tot1;
    const int64_t in0 = block_incl_sum(pk0, s_warp, &tot0);
    const int64_t in1 = block_incl_sum(pk1, s_warp, &tot1);
#pragma unroll
    for (int s = 0; s < 6; s++) {
        tot[s] = (int)(((s < 3 ? tot0 : tot1) >> (21 * (s % 3))) & 0x1FFFFF);
        excl[s] = (int)(((s < 3 ? in0 : in1) >> (21 * (s % 3))) & 0x1FFFFF) - my_cnt[s];
        before[s] = run;
        run += tot[s];
    }
    if (threadIdx.x < 6) cnt[layout_index(ti, tile_base, threadIdx.x)] = tot[threadIdx.x];
    if (threadIdx.x == 0) s_base = (long long)atomicAdd(hit_count, (unsigned long long)run);
    __syncthreads();
    const int64_t base = s_base;
    if (base + run > hit_cap || !active) return;      // overflow: the host falls back to the two-pass emit
#pragma unroll
    for (int s = 0; s < 6; s++) {
        if (my_cnt[s] == 0) continue;
        enumerate_stream<2>(ti, sm, s, x0, prev[s], is_end_thread, min_aa, two_T, base + before[s] + excl[s], excl[s], nullptr, nullptr, nullptr,
                            hits, (int32_t)tile, fl[s]);
    }
}


// ---- two-level scan (min_aa >= SIX_WIN_MIN_AA) --------------------------------------------------------------------------------
// k_six_scan spends ~18 instructions per base on exact stop positions, their prefix-max across threads / warps / tiles and
// the ORF tests, although a kept ORF of >= 100 residues needs >= 100 stop-free codons in a row: in random DNA one window of 32
// codons in five is stop-free, two in a row 4.7 %.  So:
//   pass A (k_six_bits)  one thread per WINDOW of 96 bases (32 codons of each of the six streams): "does stream s hold a stop in
//                        this window" -- six_masks + a residue mask, one ballot per stream; one bit per (stream, window) and the
//                        last window with a stop per (tile, stream).  The genome is read once, nothing else is remembered.
//   pass B (k_six_cand)  one warp per (tile, stream) walks the tile's 768 bits; a window with a stop that follows z stop-free
//                        windows can only close an ORF of < 32 (z + 2) codons, so exact stop positions are recomputed (six_masks
//                        on the two windows involved) for the few candidates only, tested with the same arithmetic as
//                        enumerate_stream and appended to the same hit list.  "Previous stop" needs no look-back chain: the
//                        bitmap is complete, the thread reads backwards over the per-tile summaries.
// Everything after the scan (counts -> prefix sums -> k_six_place -> k_six_aa) is shared with the single-pass scan, which
// stays for small min_aa.
#define SIX_WIN 96
#define SIX_WPT (SIX_TILE / SIX_WIN)                 // 768 windows per tile
#define SIX_WORDS (SIX_WPT / 32)                     // 24 bitmap words per (tile, stream)
#define SIX_WIN_MIN_AA 96                            // below this a candidate is every window: the single-pass scan is used
static_assert(SIX_TILE % (SIX_WIN * 32) == 0, "a tile must hold a whole number of bitmap words");

// stops of stream s inside window w of the contig (two 48-base halves), one bit per position
template <bool GEN>
__device__ __forceinline__ void window_stream_stops(const uint32_t *__restrict__ packed, const TileInfo &ti, int64_t w, int s,
                                                    const SixStops &ss, uint64_t x[2]) {
    const uint64_t rm = 0x0000249249249249ull << stream_res(s, ti.Lm3);
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int64_t xh = w * SIX_WIN + SIX_HALF * h;
        x[h] = 0;
        if (xh < ti.L) {
            SixMasks sm;
            if (s & 1) {                                   // one strand only: half the mask logic (s is uniform across the warp)
                six_masks_t<1, GEN>(packed, ti.gb, ti.L, xh, ti.cs, ss, sm);
                x[h] = pos48(sm.pm) & rm;
            } else {
                six_masks_t<2, GEN>(packed, ti.gb, ti.L, xh, ti.cs, ss, sm);
                x[h] = pos48(sm.mm) & rm;
            }
        }
    }
}

template <bool GEN>
__global__ void __launch_bounds__(256) k_six_bits(const uint32_t *__restrict__ packed, const int64_t *__restrict__ tile_base,
                                                  const int32_t *__restrict__ cid, const int64_t *__restrict__ contig_len,
                                                  const int64_t *__restrict__ contig_base, const int32_t *__restrict__ cs,
                                                  const int64_t *__restrict__ m, const int32_t *__restrict__ tile_contig,
                                                  uint32_t *__restrict__ bits, int32_t *__restrict__ last_set,
                                                  const __grid_constant__ SixStops ss) {
    __shared__ TileInfo ti;
    const int64_t tile = blockIdx.x / 3;
    const int part = blockIdx.x % 3;
    if (threadIdx.x == 0) tile_info_at(tile, tile_contig[tile], tile_base, cid, contig_len, contig_base, cs, m, ti);
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int wl = part * 256 + (int)threadIdx.x;          // window inside the tile
    const int64_t x0 = (ti.k * SIX_WPT + wl) * (int64_t)SIX_WIN;
    // "does residue class r of the plus / minus strand hold a stop in this window": tested on the nibble-spaced flags themselves
    // (position 16 g + k of a half has residue (g + k) % 3: three masked ORs per class) -- compressing them to one bit per
    // position first (pos48) was a quarter of this kernel's instructions
    uint64_t hp[3] = {0, 0, 0}, hm[3] = {0, 0, 0};
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int64_t xh = x0 + SIX_HALF * h;
        if (xh < ti.L) {
            SixMasks sm;
            six_masks<GEN>(packed, ti.gb, ti.L, xh, ti.cs, ss, sm);
#pragma unroll
            for (int r = 0; r < 3; r++) {
                hp[r] |= (sm.pm[0] & res_mask(r)) | (sm.pm[1] & res_mask((r + 2) % 3)) | (sm.pm[2] & res_mask((r + 1) % 3));
                hm[r] |= (sm.mm[0] & res_mask(r)) | (sm.mm[1] & res_mask((r + 2) % 3)) | (sm.mm[2] & res_mask((r + 1) % 3));
            }
        }
    }
#pragma unroll
    for (int s = 0; s < 6; s++) {
        const int r = stream_res(s, ti.Lm3);
        const uint64_t v = (s & 1) ? (r == 0 ? hp[0] : (r == 1 ? hp[1] : hp[2])) : (r == 0 ? hm[0] : (r == 1 ? hm[1] : hm[2]));
        const bool has = ti.m[s] > 0 && v != 0;
        const unsigned int b = __ballot_sync(0xffffffffu, has);
        if (lane == 0) {
            bits[(tile * 6 + s) * SIX_WORDS + part * 8 + wid] = b;
            if (b) atomicMax(last_set + tile * 6 + s, part * 256 + wid * 32 + 31 - __clz(b));
        }
    }
}

// 3 * residues of the candidate ORF between a lower stop xl and a higher stop xh (the arithmetic of enumerate_stream::visit)
__device__ __forceinline__ int64_t six_span3(const TileInfo &ti, int s, int64_t xl, bool xl_real, int64_t xh, bool xh_real) {
    const int plus = s & 1;
    const int32_t L32 = (int32_t)ti.L, cs32 = ti.cs[s], m32 = (int32_t)ti.m[s];
    const int32_t ql = plus ? (int32_t)xl - cs32 : L32 - 3 - cs32 - (int32_t)xl;
    const int32_t qh = plus ? (int32_t)xh - cs32 : L32 - 3 - cs32 - (int32_t)xh;
    if (plus) return (int64_t)(xh_real ? qh : 3 * m32) - (xl_real ? ql : -3) - 3;
    return (int64_t)(xl_real ? ql : 3 * m32) - (xh_real ? qh : -3) - 3;
}

// ---- stop-codon index ---------------------------------------------------------------------------------------------------
// The stop flags of a base depend on the genome alone (codon at t on the plus strand: TAA TAG TGA; on the minus strand: the
// reverse complements; the first-codon trims of the reference's frame quirk are per-contig constants), so they are computed ONCE
// per packed genome -- like the reverse-complement plane -- into two dense bit planes, 2 bits per base (0.25 B/base next to the
// 1 B/base of the two nibble planes).  The two-level scan then reads 0.25 B/base instead of 0.5 and spends ~1 instruction per 3
// bases instead of ~8 per base on the codon logic (k_six_bits: 790 M warp instructions, 1.08 ms on config 5).  Built lazily by
// the first ORF scan after mg_genome_finalize / mg_genome_mask (k_stop_index, one thread per 96-base window, six_masks as in the
// scan kernels, so the validity rules at contig ends are the same code).
template <bool GEN>
__global__ void __launch_bounds__(256) k_stop_index(const uint32_t *__restrict__ packed, const int64_t *__restrict__ contig_len,
                                                    const int64_t *__restrict__ contig_base, const int64_t *__restrict__ win_base, int64_t nc,
                                                    const int32_t *__restrict__ cs, uint32_t *__restrict__ sp, uint32_t *__restrict__ sm_,
                                                    const __grid_constant__ SixStops ss) {
    const int64_t flat = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (flat >= win_base[nc]) return;
    int64_t lo = 0, hi = nc;                          // largest c with win_base[c] <= flat
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (win_base[mid] <= flat) lo = mid; else hi = mid;
    }
    const int64_t w = flat - win_base[lo], L = contig_len[lo], gb = contig_base[lo];
    int32_t cs6[6];
#pragma unroll
    for (int k = 0; k < 6; k++) cs6[k] = cs[lo * 6 + k];
    uint64_t P[2] = {0, 0}, M[2] = {0, 0};
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int64_t xh = w * SIX_WIN + SIX_HALF * h;
        if (xh < L) {
            SixMasks s;
            six_masks<GEN>(packed, gb, L, xh, cs6, ss, s);
            P[h] = pos48(s.pm);
            M[h] = pos48(s.mm);
        }
    }
    const int64_t base = (gb >> 5) + 3 * w;
    const uint32_t pw[3] = {(uint32_t)P[0], (uint32_t)(P[0] >> 32) | (uint32_t)(P[1] << 16), (uint32_t)(P[1] >> 16)};
    const uint32_t mw[3] = {(uint32_t)M[0], (uint32_t)(M[0] >> 32) | (uint32_t)(M[1] << 16), (uint32_t)(M[1] >> 16)};
#pragma unroll
    for (int j = 0; j < 3; j++)
        if (w * SIX_WIN + 32 * j < L) { sp[base + j] = pw[j]; sm_[base + j] = mw[j]; }   // the words beyond belong to the next contig
}

// stops of stream s in window w of the contig from the index: three words, bit k of word j = position 96 w + 32 j + k
__device__ __forceinline__ void window_stops_ix(const uint32_t *__restrict__ stops, int64_t stop_words, const TileInfo &ti, int64_t w, int s,
                                                uint32_t x[3]) {
    const uint32_t *pl = stops + ((s & 1) ? 0 : stop_words) + (ti.gb >> 5) + 3 * w;
    const int r = stream_res(s, ti.Lm3);
#pragma unroll
    for (int j = 0; j < 3; j++) {                     // position 32 j + k of the window has residue (2 j + k) % 3
        const uint32_t rm = 0x49249249u << ((r + j) % 3);
        x[j] = w * SIX_WIN + 32 * j < ti.L ? __ldg(pl + j) & rm : 0u;
    }
}

__global__ void __launch_bounds__(256) k_six_bits_ix(const uint32_t *__restrict__ stops, int64_t stop_words, const int64_t *__restrict__ tile_base,
                                                     const int32_t *__restrict__ cid, const int64_t *__restrict__ contig_len,
                                                     const int64_t *__restrict__ contig_base, const int32_t *__restrict__ cs,
                                                     const int64_t *__restrict__ m, const int32_t *__restrict__ tile_contig,
                                                     uint32_t *__restrict__ bits, int32_t *__restrict__ last_set) {
    // one block per tile, three windows per thread (their loads are independent): the per-block prologue (tile -> contig ->
    // geometry, three dependent loads) is paid once per 768 windows
    __shared__ TileInfo ti;
    __shared__ int s_last[6];
    const int64_t tile = blockIdx.x;
    if (threadIdx.x == 0) tile_info_at(tile, tile_contig[tile], tile_base, cid, contig_len, contig_base, cs, m, ti);
    if (threadIdx.x < 6) s_last[threadIdx.x] = -1;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t p[3][3], q[3][3];
#pragma unroll
    for (int part = 0; part < 3; part++) {
        const int64_t w = ti.k * SIX_WPT + part * 256 + (int)threadIdx.x;      // window of the contig
        const int64_t base = (ti.gb >> 5) + 3 * w;
#pragma unroll
        for (int j = 0; j < 3; j++) {
            const bool in = w * SIX_WIN + 32 * j < ti.L;
            p[part][j] = in ? __ldg(stops + base + j) : 0u;
            q[part][j] = in ? __ldg(stops + stop_words + base + j) : 0u;
        }
    }
#pragma unroll
    for (int s = 0; s < 6; s++) {
        const int r = stream_res(s, ti.Lm3);
        const uint32_t r0 = 0x49249249u << r, r1 = 0x49249249u << ((r + 1) % 3), r2 = 0x49249249u << ((r + 2) % 3);
        int last = -1;
#pragma unroll
        for (int part = 0; part < 3; part++) {
            const uint32_t v = (s & 1) ? ((p[part][0] & r0) | (p[part][1] & r1) | (p[part][2] & r2))
                                       : ((q[part][0] & r0) | (q[part][1] & r1) | (q[part][2] & r2));
            const unsigned int b = __ballot_sync(0xffffffffu, ti.m[s] > 0 && v != 0);
            if (lane == 0) bits[(tile * 6 + s) * SIX_WORDS + part * 8 + wid] = b;
            if (b) last = part * 256 + wid * 32 + 31 - __clz(b);
        }
        if (lane == 0 && last >= 0) atomicMax(&s_last[s], last);
    }
    __syncthreads();
    if (threadIdx.x < 6) last_set[tile * 6 + threadIdx.x] = s_last[threadIdx.x];
}

// One WARP per (tile, stream).  Lane j holds word j of the row's bitmap (SIX_WORDS = 24 of the 32 lanes).  A window is a
// candidate only if the two windows in front of it are stop-free (one AND of shifted words; min_aa >= SIX_WIN_MIN_AA = 96 needs
// at least two) and 32 (z + 2) > min_aa for its z stop-free predecessors: ~4 % of the windows at min_aa = 100, ~28 per row, but
// 0 to 5 per word.  So the lanes first LIST the row's candidates in shared memory (window, previous window with a stop), in
// ascending order through a warp scan of their counts, and then take them 32 at a time: the exact stop positions (the
// expensive part: the genome bases of two windows) are computed by all lanes at once whatever word a candidate came from.  The
// list order is the window order, so the rank of a kept ORF inside the row is a running count + a ballot prefix.
#define CAND_WARPS 8
#define CAND_LIST (SIX_WPT / 3 + 2)                  // a candidate needs two stop-free windows in front of it
// IX: exact stop positions from the stop-codon index instead of the packed bases; GEN: as in six_masks_t (IX == false only)
template <bool IX, bool GEN>
__global__ void __launch_bounds__(32 * CAND_WARPS) k_six_cand(const uint32_t *__restrict__ packed, const uint32_t *__restrict__ stops,
                                                  int64_t stop_words, const int64_t *__restrict__ tile_base,
                                                  const int32_t *__restrict__ cid, const int64_t *__restrict__ contig_len,
                                                  const int64_t *__restrict__ contig_base, const int32_t *__restrict__ cs,
                                                  const int64_t *__restrict__ m, const int32_t *__restrict__ tile_contig, int64_t n_tiles,
                                                  const uint32_t *__restrict__ bits, const int32_t *__restrict__ last_set, int64_t min_aa,
                                                  int32_t *__restrict__ cnt, SixHit *__restrict__ hits, int64_t hit_cap,
                                                  unsigned long long *hit_count, const __grid_constant__ SixStops ss) {
    // per warp: the row's candidates (window, previous window with a stop), overwritten in place by the bounding stops (xl, xh)
    __shared__ int32_t s_w[CAND_WARPS][CAND_LIST], s_pw[CAND_WARPS][CAND_LIST];
    __shared__ uint8_t s_f[CAND_WARPS][CAND_LIST];          // bit 0 xl_real, bit 1 xh_real, bit 2 kept
    __shared__ int s_tot[CAND_WARPS];
    __shared__ unsigned long long s_slot;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t i = blockIdx.x * (int64_t)CAND_WARPS + wid;
    const bool row = i < n_tiles * 6;                      // whole warp
    const int64_t tile = row ? i / 6 : 0;
    const int s = (int)(i % 6);
    TileInfo ti;
    tile_info_at(tile, tile_contig[tile], tile_base, cid, contig_len, contig_base, cs, m, ti);
    const int64_t li = layout_index(ti, tile_base, s);
    const bool live = row && ti.m[s] > 0;                  // `if translated_seq:` (genome.py:832)
    const int64_t need3 = 3 * min_aa;
    int C = 0, total = 0;
    if (live) {
        // last window with a stop before this tile (same contig, same stream): 32 tile summaries per step, backwards
        int64_t prev_tile_w = -1;
        for (int64_t t0 = tile - 1; t0 >= tile - ti.k; t0 -= 32) {
            const int64_t tt = t0 - lane;
            const int32_t ls = tt >= tile - ti.k ? last_set[tt * 6 + s] : -1;
            const unsigned int has = __ballot_sync(0xffffffffu, ls >= 0);
            if (has) {
                const int src = __ffs(has) - 1;
                const int32_t lsv = __shfl_sync(0xffffffffu, ls, src);
                prev_tile_w = (t0 - src - (tile - ti.k)) * SIX_WPT + lsv;
                break;
            }
        }
        const int64_t w0 = ti.k * SIX_WPT + lane * 32;      // contig-level index of the first window of this lane's word
        const uint32_t b = lane < SIX_WORDS ? __ldg(bits + (tile * 6 + s) * SIX_WORDS + lane) : 0u;
        // last window with a stop before this lane's word: exclusive prefix max over the lanes, then the earlier tiles
        int64_t incl = b ? w0 + 31 - __clz(b) : -1;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d && t > incl) incl = t;
        }
        int64_t prev_before = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0 || prev_before < prev_tile_w) prev_before = prev_tile_w;
        // windows with a stop whose two predecessors are stop-free (the window in front of the contig counts as a stop, like prev = -1)
        uint32_t pword = __shfl_up_sync(0xffffffffu, b, 1);
        if (lane == 0) pword = prev_before == w0 - 1 ? 0x80000000u : (prev_before == w0 - 2 ? 0x40000000u : 0u);
        const uint64_t ext = ((uint64_t)b << 32) | pword;
        const uint32_t cand = b & ~(uint32_t)((ext << 1) >> 32) & ~(uint32_t)((ext << 2) >> 32);
        // exact test on z, then the list
        uint32_t keepm = 0;
        for (uint32_t c = cand; c; c &= c - 1) {
            const int k = __ffs(c) - 1;
            const uint32_t below = b & ((1u << k) - 1u);
            const int64_t pw = below ? w0 + 31 - __clz(below) : prev_before;
            if (32 * (w0 + k - pw - 1 + 2) > min_aa) keepm |= 1u << k;    // else the ORF this window closes has < 32 (z + 2) - 1 residues
        }
        const bool tail = lane == 31 && ti.k == ti.Tc - 1 &&      // the virtual stop at the contig's high end belongs to the last tile
                          32 * ((ti.L + SIX_WIN - 1) / SIX_WIN - prev_before - 1 + 2) > min_aa;
        int off = __popc(keepm) + (tail ? 1 : 0);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, off, d);
            if (lane >= d) off += t;
        }
        C = __shfl_sync(0xffffffffu, off, 31);
        off -= __popc(keepm) + (tail ? 1 : 0);
        for (uint32_t c = keepm; c; c &= c - 1) {
            const int k = __ffs(c) - 1;
            const uint32_t below = b & ((1u << k) - 1u);
            s_w[wid][off] = (int32_t)(w0 + k);
            s_pw[wid][off] = (int32_t)(below ? w0 + 31 - __clz(below) : prev_before);
            off++;
        }
        if (tail) { s_w[wid][off] = -1; s_pw[wid][off] = (int32_t)prev_before; }
        __syncwarp();
        for (int r0 = 0; r0 < C; r0 += 32) {
            const int idx = r0 + lane;
            bool pass = false;
            if (idx < C) {
                const int64_t w = s_w[wid][idx], pw = s_pw[wid][idx];
                const bool xl_real = pw >= 0, xh_real = w >= 0;
                int64_t xl = -1, xh = 0;
                if (IX) {
                    uint32_t y[3];
                    if (xh_real) {
                        window_stops_ix(stops, stop_words, ti, w, s, y);
                        xh = w * SIX_WIN + (y[0] ? __ffs(y[0]) - 1 : (y[1] ? 32 + __ffs(y[1]) - 1 : 64 + __ffs(y[2]) - 1));
                    }
                    if (xl_real) {                         // exact position of the last stop of the stream in window pw (it has one)
                        window_stops_ix(stops, stop_words, ti, pw, s, y);
                        xl = pw * SIX_WIN + (y[2] ? 64 + 31 - __clz(y[2]) : (y[1] ? 32 + 31 - __clz(y[1]) : 31 - __clz(y[0])));
                    }
                } else {
                    uint64_t x[2];
                    if (xh_real) {
                        window_stream_stops<GEN>(packed, ti, w, s, ss, x);
                        xh = w * SIX_WIN + (x[0] ? __ffsll((long long)x[0]) - 1 : SIX_HALF + __ffsll((long long)x[1]) - 1);
                    }
                    if (xl_real) {
                        window_stream_stops<GEN>(packed, ti, pw, s, ss, x);
                        xl = pw * SIX_WIN + (x[1] ? SIX_HALF + 63 - __clzll((long long)x[1]) : 63 - __clzll((long long)x[0]));
                    }
                }
                pass = six_span3(ti, s, xl, xl_real, xh, xh_real) >= need3;
                s_w[wid][idx] = (int32_t)xl;
                s_pw[wid][idx] = (int32_t)xh;
                s_f[wid][idx] = (uint8_t)((xl_real ? 1 : 0) | (xh_real ? 2 : 0) | (pass ? 4 : 0));
            }
            total += __popc(__ballot_sync(0xffffffffu, pass));
        }
    }
    // one slot allocation per block (a quarter of a million same-address atomics, one per row, were as long as the rest of the kernel)
    if (lane == 0) s_tot[wid] = total;
    __syncthreads();
    if (threadIdx.x == 0) {
        int sum = 0;
#pragma unroll
        for (int k = 0; k < CAND_WARPS; k++) sum += s_tot[k];
        s_slot = sum ? atomicAdd(hit_count, (unsigned long long)sum) : 0ull;
    }
    __syncthreads();
    if (!row) return;
    if (!live) { if (lane == 0) cnt[li] = 0; return; }
    unsigned long long slot = s_slot;
    for (int k = 0; k < wid; k++) slot += s_tot[k];
    int rank = 0;
    for (int r0 = 0; r0 < C; r0 += 32) {
        const int idx = r0 + lane;
        const uint32_t f = idx < C ? s_f[wid][idx] : 0u;
        const unsigned int bal = __ballot_sync(0xffffffffu, (f & 4u) != 0);
        const int my = rank + __popc(bal & ((1u << lane) - 1u));
        if ((f & 4u) && (int64_t)(slot + my) < hit_cap) {
            SixHit h;
            h.tile = (int32_t)tile; h.rank = my; h.xl = s_w[wid][idx]; h.xh = s_pw[wid][idx];
            h.s = (uint8_t)s; h.xl_real = f & 1u; h.xh_real = (f >> 1) & 1u; h.pad = 0;
            hits[slot + my] = h;
        }
        rank += __popc(bal);
    }
    if (lane == 0) cnt[li] = total;
}

// thread per hit: reference-order slot of the ORF and its record
__global__ void __launch_bounds__(256) k_six_place(const SixHit *__restrict__ hits, int64_t n_hit, const int64_t *__restrict__ tile_base,
                                                   int64_t nc, const int32_t *__restrict__ cid, const int64_t *__restrict__ contig_len,
                                                   const int64_t *__restrict__ contig_base, const int32_t *__restrict__ cs,
                                                   const int64_t *__restrict__ m, const int64_t *__restrict__ cnt_off, int64_t two_T,
                                                   mg_orf *__restrict__ recs, int32_t *__restrict__ lens, int64_t *__restrict__ srcs) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_hit) return;
    const SixHit h = hits[i];
    TileInfo ti;
    tile_info(h.tile, tile_base, nc, cid, contig_len, contig_base, cs, m, ti);
    const int s = h.s, plus = s & 1;
    const int64_t li = layout_index(ti, tile_base, s);
    const int64_t o0 = cnt_off[li], n = cnt_off[li + 1] - o0;
    const int64_t slot = o0 + (plus ? h.rank : n - 1 - h.rank);
    int64_t st, ln;
    orf_of(plus, ti.L, ti.cs[s], ti.m[s], h.xl, h.xh, h.xl_real, h.xh_real, st, ln);
    mg_orf o;
    o.contig = (int32_t)ti.c; o.frame = (int8_t)(s >> 1); o.minus = (int8_t)(!plus); o.pad = 0;
    o.start = st; o.len = ln; o.aa_off = 0;
    recs[slot] = o;
    lens[slot] = (int32_t)ln;
    const int64_t q = ti.cs[s] + 3 * st;                                // oriented offset of the ORF's first base
    srcs[slot] = plus ? (ti.gb + q) : (two_T - ti.gb - ti.L + q);      // '-': forward read of the reverse plane
}

__global__ void __launch_bounds__(256) k_six_fill_off(int64_t n_orf, const int64_t *__restrict__ aa_off, mg_orf *__restrict__ recs) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n_orf) recs[i].aa_off = aa_off[i];
}

__global__ void __launch_bounds__(256) k_six_tiles(const int64_t *__restrict__ off, int64_t n, int64_t tile_bytes, int64_t n_tile,
                                                   int64_t *__restrict__ tile_first) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t > n_tile) return;
    if (t == n_tile) { tile_first[t] = n > 0 ? n - 1 : 0; return; }
    tile_first[t] = mg_search_le(off, 0, n, t * tile_bytes);
}

// ---- pass E: residues of the kept ORFs, flat over output bytes (16 per thread) ------------------------------
__global__ void __launch_bounds__(AA_THREADS) k_six_aa(const uint32_t *__restrict__ packed, const int64_t *__restrict__ aa_off,
                                                       const int64_t *__restrict__ srcs, int64_t n_orf,
                                                       const int64_t *__restrict__ tile_first, int64_t total,
                                                       const uint8_t *__restrict__ aa4096, uint8_t *__restrict__ out) {
    __shared__ __align__(16) uint8_t s_aa[4096];
    __shared__ int64_t s_off[AA_CAP + 1];             // residue offsets of the tile's ORFs ...
    __shared__ int64_t s_src[AA_CAP];                 // ... and the index of their first base (either plane, a forward read)
    reinterpret_cast<uint4 *>(s_aa)[threadIdx.x] = __ldg(reinterpret_cast<const uint4 *>(aa4096) + threadIdx.x);
    const int64_t P0 = (int64_t)blockIdx.x * AA_TILE;
    const int64_t o_lo = tile_first[blockIdx.x];
    int64_t o_hi = tile_first[blockIdx.x + 1] + 1;
    if (o_hi > n_orf) o_hi = n_orf;
    const int ncache = (int)min((int64_t)AA_CAP, o_hi - o_lo);
    for (int i = threadIdx.x; i <= ncache; i += AA_THREADS) {
        s_off[i] = __ldg(aa_off + o_lo + i);
        if (i < ncache) s_src[i] = __ldg(srcs + o_lo + i);
    }
    __syncthreads();
    const int64_t cached_end = s_off[ncache];
#pragma unroll 1
    for (int cidx = 0; cidx < AA_TILE / 16 / AA_THREADS; cidx++) {
        const int64_t P = P0 + ((int64_t)(cidx * AA_THREADS + threadIdx.x) << 4);
        if (P >= total) break;
        uint64_t blo = 0, bhi = 0;
        int filled = 0;
        int64_t pos = P;
        if (P + 16 <= cached_end) {
            // the whole chunk lies in ORFs staged in shared memory (always, unless a tile holds more than AA_CAP ORFs)
            int lo = 0, hi = ncache;
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (s_off[mid] <= P) lo = mid; else hi = mid;
            }
            uint32_t bw[4] = {0, 0, 0, 0};
            const int64_t left = s_off[lo + 1] - P;   // residues of ORF lo from P on
            if (left >= 16 || s_off[lo + 2] >= P + 16) {
                // One or two ORFs in the chunk (always, for min_aa >= 16): their nibbles are merged BEFORE the look-ups, as K2 merges
                // two pieces -- the second ORF's window is fetched at an index chosen so that its first base lands on window nibble
                // 3c -- so no lane takes a second trip (the per-ORF loop below ran at 15 of 32 lanes: 72 % of the warps hold a
                // chunk with an ORF boundary) and the 16 look-ups are done once.
                const int c = left >= 16 ? 16 : (int)left;
                const int64_t g0 = s_src[lo] + 3 * (P - s_off[lo]);
                const int64_t g1 = (c < 16 ? s_src[lo + 1] : g0 + 48) - 3 * c;
                const uint32_t *pa = packed + (g0 >> 3), *pb = packed + (g1 >> 3);
                const uint32_t sha = ((uint32_t)g0 & 7u) << 2, shb = ((uint32_t)g1 & 7u) << 2;
                uint32_t va[7], vb[7], n[6];
#pragma unroll
                for (int k = 0; k < 7; k++) { va[k] = __ldg(pa + k); vb[k] = __ldg(pb + k); }
#pragma unroll
                for (int k = 0; k < 6; k++) {
                    const int t = 3 * c - 8 * k;                                   // window nibbles < 3c come from the first ORF
                    const uint32_t m = __funnelshift_lc(0xFFFFFFFFu, 0u, (uint32_t)(4 * max(t, 0)));
                    n[k] = (__funnelshift_r(va[k], va[k + 1], sha) & m) | (__funnelshift_r(vb[k], vb[k + 1], shb) & ~m);
                }
#pragma unroll
                for (int k = 0; k < 16; k++) {            // codon k = nibbles 3k..3k+2 = bits 12k.. of n[5]:..:n[0]
                    const int bit = 12 * k, ww = bit >> 5, sh = bit & 31;
                    uint32_t idx = n[ww] >> sh;
                    if (sh > 20) idx |= n[ww + 1] << (32 - sh);
                    bw[k >> 2] |= (uint32_t)s_aa[idx & 0xFFFu] << ((k & 3) * 8);
                }
                filled = 16;
            }
            while (filled < 16 && pos < total) {
                while (s_off[lo + 1] <= pos) lo++;
                const int64_t a = pos - s_off[lo];
                int c = 16 - filled;
                if (s_off[lo + 1] - pos < c) c = (int)(s_off[lo + 1] - pos);
                // 16 codons = 48 nibbles from one ORF: seven words, six funnel shifts (as K3), then 12-bit table indices
                const int64_t g0 = s_src[lo] + 3 * a;
                const uint32_t *pp = packed + (g0 >> 3);
                const uint32_t sh0 = ((uint32_t)g0 & 7u) << 2;
                uint32_t v[7], n[6];
#pragma unroll
                for (int k = 0; k < 7; k++) v[k] = __ldg(pp + k);
#pragma unroll
                for (int k = 0; k < 6; k++) n[k] = __funnelshift_r(v[k], v[k + 1], sh0);
                uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
                for (int k = 0; k < 16; k++) {            // codon k = nibbles 3k..3k+2 = bits 12k.. of n[5]:..:n[0]
                    const int bit = 12 * k, ww = bit >> 5, sh = bit & 31;
                    uint32_t idx = n[ww] >> sh;
                    if (sh > 20) idx |= n[ww + 1] << (32 - sh);
                    w[k >> 2] |= (uint32_t)s_aa[idx & 0xFFFu] << ((k & 3) * 8);
                }
                if (c == 16) { bw[0] = w[0]; bw[1] = w[1]; bw[2] = w[2]; bw[3] = w[3]; }
                else {                                    // c residues of this ORF land at chunk positions [filled, filled + c)
                    const uint32_t m = ((1u << c) - 1u);
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        // shift the c residues up by `filled` bytes inside the 16-byte chunk
                        uint32_t lo32 = 0;
                        const int byte0 = 4 * k - filled;     // source byte that lands on byte 4k
#pragma unroll
                        for (int b = 0; b < 4; b++) {
                            const int sb = byte0 + b;
                            if (sb >= 0 && sb < 16 && ((m >> sb) & 1u)) lo32 |= ((w[sb >> 2] >> ((sb & 3) * 8)) & 0xFFu) << (8 * b);
                        }
                        bw[k] |= lo32;
                    }
                }
                filled += c;
                pos += c;
            }
            blo = ((uint64_t)bw[1] << 32) | bw[0];
            bhi = ((uint64_t)bw[3] << 32) | bw[2];
        } else {
            int64_t o = P < cached_end ? o_lo : o_lo + ncache;
            o = mg_search_le(aa_off, o, n_orf, P);
            int64_t off_o = __ldg(aa_off + o), off_n = __ldg(aa_off + o + 1);
            while (filled < 16 && pos < total) {
                while (off_n <= pos) { o++; off_o = off_n; off_n = __ldg(aa_off + o + 1); }
                const int64_t a = pos - off_o;
                int c = 16 - filled;
                if (off_n - pos < c) c = (int)(off_n - pos);
                const int64_t g0 = __ldg(srcs + o) + 3 * a;      // either plane, always a forward read
                uint64_t acc[3];
                acc[0] = mg_ld_nib16(packed, g0);
                acc[1] = mg_ld_nib16(packed, g0 + 16);
                acc[2] = mg_ld_nib16(packed, g0 + 32);
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    if (k < c) {
                        const int bit = 12 * k, w = bit >> 6, sh = bit & 63;
                        uint32_t idx = (uint32_t)(acc[w] >> sh);
                        if (sh > 52) idx |= (uint32_t)(acc[w + 1] << (64 - sh));
                        const uint64_t b = s_aa[idx & 0xFFFu];
                        const int t = filled + k;
                        if (t < 8) blo |= b << (8 * t); else bhi |= b << (8 * (t - 8));
                    }
                }
                filled += c;
                pos += c;
            }
        }
        mg_st16(out + P, (uint32_t)blo, (uint32_t)(blo >> 32), (uint32_t)bhi, (uint32_t)(bhi >> 32));
    }
}

// ---- ORF calling (mg_orfcall_count): start codon of each stop-bounded segment -----------------------------------------
// The scan kernels above, run on the true-phase geometry (k_orf_streams) with min_aa as the segment threshold, place every
// segment of >= min_aa codons (an ORF never outruns its segment).  k_orf_start finds each segment's first start codon,
// mg_scan_i32 compacts the kept ones, k_orf_place writes their records, and k_six_aa + k_orf_first_m their residues.
#define ORF_WARPS 8
#define ORF_SPAN 512                                  // codons a warp tests per step: 16 per lane, one 48-nibble window each

// One WARP per segment, ORF_SPAN codons per step from the segment's first base (srcs: a forward read of either plane), until
// the first start codon: a segment of n codons costs ceil(n_to_first_start / 512) steps, so a stop-free stretch of any length
// never holds one lane for long.  kpos = codon offset of the start (-1: none); keep = start found, len - kpos >= min_aa and a
// real stop ends the segment (or partial).
__global__ void __launch_bounds__(32 * ORF_WARPS) k_orf_start(const uint32_t *__restrict__ packed, const mg_orf *__restrict__ segs,
                                                              const int64_t *__restrict__ srcs, int64_t n_seg,
                                                              const int64_t *__restrict__ contig_len, const uint8_t *__restrict__ start4096,
                                                              int64_t min_aa, int partial, int32_t *__restrict__ kpos,
                                                              int32_t *__restrict__ keep) {
    __shared__ __align__(16) uint8_t s_st[4096];
    for (int k = threadIdx.x; k < 256; k += blockDim.x)
        reinterpret_cast<uint4 *>(s_st)[k] = __ldg(reinterpret_cast<const uint4 *>(start4096) + k);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t i = blockIdx.x * (int64_t)ORF_WARPS + (threadIdx.x >> 5);
    if (i >= n_seg) return;                           // whole warp
    const int64_t len = segs[i].len, src = srcs[i];
    int64_t found = -1;
    for (int64_t base = 0; base < len && found < 0; base += ORF_SPAN) {
        const int64_t c0 = base + 16 * lane;
        uint32_t hits = 0;
        if (c0 < len) {
            const int64_t g0 = src + 3 * c0;
            const uint32_t *pp = packed + (g0 >> 3);
            const uint32_t sh0 = ((uint32_t)g0 & 7u) << 2;
            uint32_t v[7], n[6];
#pragma unroll
            for (int k = 0; k < 7; k++) v[k] = __ldg(pp + k);
#pragma unroll
            for (int k = 0; k < 6; k++) n[k] = __funnelshift_r(v[k], v[k + 1], sh0);
#pragma unroll
            for (int k = 0; k < 16; k++) {            // codon k = nibbles 3k..3k+2 = bits 12k.. of n[5]:..:n[0]
                const int bit = 12 * k, ww = bit >> 5, sh = bit & 31;
                uint32_t idx = n[ww] >> sh;
                if (sh > 20) idx |= n[ww + 1] << (32 - sh);
                hits |= (s_st[idx & 0xFFFu] != 0 ? 1u : 0u) << k;
            }
            if (len - c0 < 16) hits &= (1u << (len - c0)) - 1u;
        }
        const unsigned int any = __ballot_sync(0xffffffffu, hits != 0);
        if (any) {
            const int l = __ffs(any) - 1;
            found = base + 16 * l + __ffs(__shfl_sync(0xffffffffu, hits, l)) - 1;
        }
    }
    if (lane == 0) {
        const mg_orf o = segs[i];
        const int f = o.frame, phase = f == 0 ? 0 : (f == 1 ? 2 : 1);
        const int64_t L = contig_len[o.contig], m = L > phase ? (L - phase) / 3 : 0;
        const bool stop = o.start + len < m;          // else the segment ends at the contig end
        kpos[i] = (int32_t)found;
        keep[i] = found >= 0 && len - found >= min_aa && (stop || partial);
    }
}

// thread per segment: the kept ones' records, residue counts and first bases, compacted in segment order
__global__ void __launch_bounds__(256) k_orf_place(const uint32_t *__restrict__ packed, const mg_orf *__restrict__ segs,
                                                   const int64_t *__restrict__ srcs, int64_t n_seg, const int64_t *__restrict__ contig_len,
                                                   const uint8_t *__restrict__ start4096, const int32_t *__restrict__ kpos,
                                                   const int32_t *__restrict__ keep, const int64_t *__restrict__ slot,
                                                   mg_orfcall *__restrict__ calls, int32_t *__restrict__ lens, int64_t *__restrict__ srcs_out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_seg || !keep[i]) return;
    const mg_orf o = segs[i];
    const int64_t j = slot[i], k = kpos[i];
    const int f = o.frame, phase = f == 0 ? 0 : (f == 1 ? 2 : 1);
    const int64_t L = contig_len[o.contig], m = L > phase ? (L - phase) / 3 : 0;
    const bool stop = o.start + o.len < m;
    const int64_t len = o.len - k, g = srcs[i] + 3 * k;
    const int64_t q = phase + 3 * (o.start + k);      // oriented offset of the start codon
    const int64_t span = 3 * len + (stop ? 3 : 0);
    mg_orfcall c;
    c.contig = o.contig; c.minus = o.minus; c.phase = (int8_t)phase; c.flags = stop ? 0 : 1;
    c.start_codon = (int8_t)(start4096[mg_ld_nib16(packed, g) & 0xFFFu] - 1);
    c.lo = o.minus ? L - q - span : q;
    c.hi = c.lo + span;
    c.len = len;
    c.aa_off = 0;
    calls[j] = c;
    lens[j] = (int32_t)len;
    srcs_out[j] = g;
}

__global__ void __launch_bounds__(256) k_orf_fill_off(int64_t n, const int64_t *__restrict__ aa_off, mg_orfcall *__restrict__ calls) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) calls[i].aa_off = aa_off[i];
}

// after k_six_aa: every ORF's first residue is M, whatever its start codon
__global__ void __launch_bounds__(256) k_orf_first_m(int64_t n, const int64_t *__restrict__ aa_off, uint8_t *__restrict__ out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) out[aa_off[i]] = 'M';
}

// Start flags indexed like build_aa4096's residue table (12-bit nibble triplet), by the same decoding: 1 + codon index for a
// start codon, 0 for any other triplet (a base outside ACGT included).
static void build_start4096(uint8_t *t, const uint8_t *start64) {
    uint8_t c64[64];
    for (int c = 0; c < 64; c++) c64[c] = start64[c] ? (uint8_t)(1 + c) : 0;
    build_aa4096(t, c64);
    for (int i = 0; i < 4096; i++)
        if (t[i] == 'X') t[i] = 0;                   // 'X' (88) is no 1 + codon index (1..64)
}

// ---- host API -------------------------------------------------------------------------------------------------
static void six_release(mg_sixframe_state *s) {
    for (void *d : s->owned) cudaFreeAsync(d, s->stream);
    s->owned.clear();
    if (s->d_aa) cudaFree(s->d_aa);
    s->d_aa = nullptr;
    s->aa_cap = 0;
}

void mg_sixframe_free(mg_genome *g) {
    if (g->six) {
        six_release(g->six);
        delete g->six;
        g->six = nullptr;
    }
}

template <typename T>
static int six_alloc(mg_sixframe_state *s, T **p, int64_t n) {
    void *d = nullptr;                               // stream-ordered pool: no device-wide sync per allocation
    MG_CUDA(cudaMallocAsync(&d, std::max<int64_t>(1, n) * sizeof(T), s->stream));
    s->owned.push_back(d);
    *p = (T *)d;
    return MG_OK;
}

// stop-codon index of the whole genome (see k_stop_index) for the stop set `key` (bit 16*b0 + 4*b1 + b2 per stop codon);
// st-ordered, no host wait.  The standard set has its own index; ONE other set is kept next to it (0.25 B/base more), so
// that scans with another genetic code neither rebuild nor overwrite the standard one.  *out = the index to scan.
static int six_build_stops(mg_genome *g, cudaStream_t st, uint64_t key, const SixStops &ss, const uint32_t **out) {
    const bool gen = key != SIX_STD_STOPS;
    uint32_t *&buf = gen ? g->d_stops_alt : g->d_stops;
    *out = buf;
    if (gen ? (g->stops_alt_valid && g->stops_alt_key == key) : g->stops_valid) return MG_OK;
    const int64_t W = g->total_bases / 32 + 8, nc = g->n_contigs;
    if (!buf) {                                              // W only depends on the genome's size, fixed at mg_genome_create
        MG_CUDA(cudaMalloc((void **)&buf, 2 * W * sizeof(uint32_t)));
        g->stop_words = W;
        g->device_bytes += 2 * W * 4;
    }
    *out = buf;
    if (gen) { g->stops_alt_valid = false; g->stops_alt_key = key; }
    MG_CUDA(cudaMemsetAsync(buf, 0, 2 * W * sizeof(uint32_t), st));
    std::vector<int64_t> wb(nc + 1, 0);
    std::vector<int32_t> ident(nc);
    for (int64_t c = 0; c < nc; c++) { wb[c + 1] = wb[c] + (g->h_contig_len[c] + SIX_WIN - 1) / SIX_WIN; ident[c] = (int32_t)c; }
    if (wb[nc] == 0) { (gen ? g->stops_alt_valid : g->stops_valid) = true; return MG_OK; }
    char *tmp = nullptr;                                     // win_base | cs | m | ident
    const size_t o_cs = (nc + 1) * 8, o_m = o_cs + nc * 6 * 4 + 8, o_id = o_m + nc * 6 * 8, bytes = o_id + nc * 4;
    MG_CUDA(cudaMallocAsync((void **)&tmp, bytes, st));
    int64_t *d_wb = (int64_t *)tmp, *d_m = (int64_t *)(tmp + (o_m & ~(size_t)7));
    int32_t *d_cs = (int32_t *)(tmp + o_cs), *d_id = (int32_t *)(tmp + o_id);
    MG_CUDA(cudaMemcpyAsync(d_wb, wb.data(), (nc + 1) * 8, cudaMemcpyHostToDevice, st));
    MG_CUDA(cudaMemcpyAsync(d_id, ident.data(), nc * 4, cudaMemcpyHostToDevice, st));
    k_six_streams<<<(unsigned)((nc * 6 + 127) / 128), 128, 0, st>>>(g->d_packed, g->d_contig_len, g->d_contig_base, d_id, nc, d_cs, d_m);
    MG_LAUNCH_CHECK();
    (gen ? k_stop_index<true> : k_stop_index<false>)<<<(unsigned)((wb[nc] + 255) / 256), 256, 0, st>>>(
        g->d_packed, g->d_contig_len, g->d_contig_base, d_wb, nc, d_cs, buf, buf + W, ss);
    MG_LAUNCH_CHECK();
    MG_CUDA(cudaStreamSynchronize(st));                      // wb / ident are host vectors of this frame
    MG_CUDA(cudaFreeAsync(tmp, st));
    (gen ? g->stops_alt_valid : g->stops_valid) = true;
    return MG_OK;
}

// ORF calling after the scan placed the n_orf segments: their start codons, the kept ones compacted into d_calls / d_len / d_src
// (which then describe the ORFs, not the segments), s->n_orf = their number.
static int orf_select(mg_genome *g, mg_sixframe_state *s, const uint8_t *start64, int partial, int64_t min_aa) {
    cudaStream_t st = s->stream;
    const int64_t n_seg = s->n_orf;
    int rc;
#define TRY(x) do { rc = (x); if (rc) return rc; } while (0)
    build_start4096(s->h_start4096, start64);
    TRY(six_alloc(s, &s->d_start4096, 4096));
    MG_CUDA(cudaMemcpyAsync(s->d_start4096, s->h_start4096, 4096, cudaMemcpyHostToDevice, st));
    int32_t *d_k = nullptr, *d_keep = nullptr, *d_len = nullptr;
    int64_t *d_slot = nullptr, *d_src = nullptr;
    TRY(six_alloc(s, &d_k, n_seg));
    TRY(six_alloc(s, &d_keep, n_seg));
    TRY(six_alloc(s, &d_slot, n_seg + 1));
    k_orf_start<<<(unsigned)((n_seg + ORF_WARPS - 1) / ORF_WARPS), 32 * ORF_WARPS, 0, st>>>(
        g->d_packed, s->d_recs, s->d_src, n_seg, g->d_contig_len, s->d_start4096, min_aa, partial, d_k, d_keep);
    MG_LAUNCH_CHECK();
    const int64_t need = mg_scan_tmp_elems(n_seg) + 2;
    if (need > s->scan_tmp_cap) {
        TRY(six_alloc(s, &s->d_scan_tmp, need));
        s->scan_tmp_cap = need;
    }
    TRY(mg_scan_i32(d_keep, d_slot, n_seg, s->d_scan_tmp, s->scan_tmp_cap, st));
    // records for up to n_seg ORFs, so that k_orf_place runs before the host knows how many are kept
    TRY(six_alloc(s, &s->d_calls, n_seg));
    TRY(six_alloc(s, &d_len, n_seg));
    TRY(six_alloc(s, &d_src, n_seg));
    k_orf_place<<<(unsigned)((n_seg + 255) / 256), 256, 0, st>>>(g->d_packed, s->d_recs, s->d_src, n_seg, g->d_contig_len, s->d_start4096,
                                                                  d_k, d_keep, d_slot, s->d_calls, d_len, d_src);
    MG_LAUNCH_CHECK();
    MG_CUDA(cudaMemcpyAsync(&s->n_orf, d_slot + n_seg, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MG_CUDA(cudaStreamSynchronize(st));
    s->d_len = d_len;
    s->d_src = d_src;
#undef TRY
    return MG_OK;
}

// the arguments of mg_orfcall_count that the scan does not use (orf == NULL in six_count: the six-frame scan)
struct OrfSel {
    const uint8_t *start64;
    int partial;
};

static int six_validate(mg_genome *g, int64_t n_list, const int64_t *contig_ids, int64_t min_aa, const uint8_t *codon64) {
    MG_REQUIRE(g != nullptr, "genome handle is NULL");
    MG_REQUIRE(g->finalized, "mg_genome_finalize has not been called");
    MG_REQUIRE(n_list >= 0 && (n_list == 0 || contig_ids != nullptr), "bad contig list");
    MG_REQUIRE(min_aa >= 0, "min_aa must be >= 0");
    for (int64_t i = 0; i < n_list; i++) MG_REQUIRE(contig_ids[i] >= 0 && contig_ids[i] < g->n_contigs, "contig index out of range");
    // k_six_streams drops a leading codon for trimX when it holds a base outside ACGT, i.e. where the table gives 'X'
    if (codon64)
        for (int c = 0; c < 64; c++) MG_REQUIRE(codon64[c] != 'X', "codon64 maps an A/C/G/T codon to 'X'");
    return MG_OK;
}

// Both scans.  orf == NULL: the six-frame ORF list (the reference's geometry).  Otherwise ORF calling: the true-phase geometry,
// then the start-codon selection of the placed segments.  The stop-codon index serves both geometries unchanged: six_masks
// reads the geometry only to clear the first codon of a trimmed stream, and a codon with a base outside ACGT is never a stop.
static int six_count(mg_genome *g, int64_t n_list, const int64_t *contig_ids, int64_t min_aa, const uint8_t *codon64,
                     const OrfSel *orf, int64_t *n_orf, int64_t *n_bytes, void *stream) {
    // the genetic code: its stop set selects the scan kernels, its table the residues
    uint64_t key = SIX_STD_STOPS;
    SixStops ss;
    memset(&ss, 0, sizeof(ss));
    if (codon64) {
        key = 0;
        for (int c = 0; c < 64; c++) {
            if (codon64[c] != '*') continue;
            key |= 1ull << c;
            ss.fwd[ss.n] = (uint8_t)c;
            ss.rev[ss.n] = (uint8_t)(16 * (3 - (c & 3)) + 4 * (3 - ((c >> 2) & 3)) + (3 - (c >> 4)));
            ss.n++;
        }
    }
    const bool gen = key != SIX_STD_STOPS;
    MG_CUDA(cudaSetDevice(g->device));
    cudaStream_t st = (cudaStream_t)stream;
    mg_sixframe_free(g);
    mg_sixframe_state *s = new mg_sixframe_state();
    g->six = s;
    s->stream = st;
    s->min_aa = min_aa;
    s->force_single = g_six_force_single;
    s->orfcall = orf != nullptr;
    s->generation = g->generation;
    const int64_t nc = n_list;
    std::vector<int32_t> &h_cid = s->h_cid;
    h_cid.resize(nc);
    for (int64_t i = 0; i < nc; i++) h_cid[i] = (int32_t)contig_ids[i];
    s->h_tile_base.assign(nc + 1, 0);
    for (int64_t c = 0; c < nc; c++) {
        const int64_t L = g->h_contig_len[h_cid[c]];
        MG_REQUIRE(L < (1ll << 31), "contigs of 2^31 bases or more are not supported by the ORF scan");
        s->h_tile_base[c + 1] = s->h_tile_base[c] + (L + SIX_TILE - 1) / SIX_TILE;
    }
    s->n_tiles = s->h_tile_base[nc];
    s->n_orf = 0;
    s->n_bytes = 0;
    s->counted = true;
    if (n_orf) *n_orf = 0;
    if (n_bytes) *n_bytes = 0;
    if (s->n_tiles == 0) return MG_OK;
    int rc;
#define TRY(x) do { rc = (x); if (rc) return rc; } while (0)
    if (codon64) {
        build_aa4096(s->h_aa4096, codon64);
        TRY(six_alloc(s, &s->d_aa4096, 4096));
        MG_CUDA(cudaMemcpyAsync(s->d_aa4096, s->h_aa4096, 4096, cudaMemcpyHostToDevice, st));
    }
    TRY(six_alloc(s, &s->d_cid, nc));
    MG_CUDA(cudaMemcpyAsync(s->d_cid, h_cid.data(), nc * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    TRY(six_alloc(s, &s->d_tile_base, nc + 1));
    MG_CUDA(cudaMemcpyAsync(s->d_tile_base, s->h_tile_base.data(), (nc + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    TRY(six_alloc(s, &s->d_cs, nc * 6));
    TRY(six_alloc(s, &s->d_m, nc * 6));
    TRY(six_alloc(s, &s->d_carry, s->n_tiles * 6));
    TRY(six_alloc(s, &s->d_cnt, s->n_tiles * 6));
    TRY(six_alloc(s, &s->d_cnt_off, s->n_tiles * 6 + 1));
    TRY(six_alloc(s, &s->d_look, 6 * s->n_tiles + 2));
    s->d_hit_count = s->d_look + 6 * s->n_tiles + 1;
    s->hit_cap = std::max<int64_t>(1 << 16, s->n_tiles * (SIX_TILE / 512));   // one kept ORF per 512 bases; more: two-pass emit
    if (const char *e = getenv("MG_SIX_HIT_CAP")) s->hit_cap = std::max<int64_t>(1, atoll(e));   // tests force the second pass
    TRY(six_alloc(s, &s->d_hits, s->hit_cap));
    MG_CUDA(cudaMemsetAsync(s->d_look, 0, (6 * s->n_tiles + 2) * sizeof(unsigned long long), st));
    if (orf) k_orf_streams<<<(unsigned)((nc * 6 + 127) / 128), 128, 0, st>>>(g->d_contig_len, s->d_cid, nc, s->d_cs, s->d_m);
    else k_six_streams<<<(unsigned)((nc * 6 + 127) / 128), 128, 0, st>>>(g->d_packed, g->d_contig_len, g->d_contig_base, s->d_cid, nc, s->d_cs, s->d_m);
    MG_LAUNCH_CHECK();
    TRY(six_alloc(s, &s->d_tile_contig, s->n_tiles));
    k_six_tile_contig<<<(unsigned)((s->n_tiles + 255) / 256), 256, 0, st>>>(s->d_tile_base, nc, s->n_tiles, s->d_tile_contig);
    MG_LAUNCH_CHECK();
    // min_aa >= 96: two-level scan over the stop-codon index (MAGOT_SIX=single forces the single pass over the packed bases,
    // MAGOT_SIX=bases the two-level scan with the codon logic on the packed bases; A/B knobs)
    if (g_six_mode < 0) { const char *e = getenv("MAGOT_SIX"); g_six_mode = (e && !strcmp(e, "single")) ? 0 : ((e && !strcmp(e, "bases")) ? 1 : 2); }
    const int two_level = g_six_mode;
    const bool use_two_level = two_level && min_aa >= SIX_WIN_MIN_AA && !s->force_single;
    if (use_two_level) {
        uint32_t *d_bits = nullptr;
        int32_t *d_last = nullptr;
        TRY(six_alloc(s, &d_bits, s->n_tiles * 6 * SIX_WORDS));
        TRY(six_alloc(s, &d_last, s->n_tiles * 6));
        MG_CUDA(cudaMemsetAsync(d_last, 0xFF, s->n_tiles * 6 * sizeof(int32_t), st));
        const unsigned cand_grid = (unsigned)((s->n_tiles * 6 + CAND_WARPS - 1) / CAND_WARPS);
        if (two_level == 2) {
            const uint32_t *stops = nullptr;
            TRY(six_build_stops(g, st, key, ss, &stops));
            k_six_bits_ix<<<(unsigned)s->n_tiles, 256, 0, st>>>(stops, g->stop_words, s->d_tile_base, s->d_cid, g->d_contig_len,
                                                                     g->d_contig_base, s->d_cs, s->d_m, s->d_tile_contig, d_bits, d_last);
            MG_LAUNCH_CHECK();
            k_six_cand<true, false><<<cand_grid, 32 * CAND_WARPS, 0, st>>>(g->d_packed, stops, g->stop_words, s->d_tile_base, s->d_cid,
                                                                            g->d_contig_len, g->d_contig_base, s->d_cs, s->d_m, s->d_tile_contig,
                                                                            s->n_tiles, d_bits, d_last, min_aa, s->d_cnt, s->d_hits, s->hit_cap,
                                                                            s->d_hit_count, ss);
            MG_LAUNCH_CHECK();
        } else {
            (gen ? k_six_bits<true> : k_six_bits<false>)<<<(unsigned)(s->n_tiles * 3), 256, 0, st>>>(
                g->d_packed, s->d_tile_base, s->d_cid, g->d_contig_len, g->d_contig_base, s->d_cs, s->d_m, s->d_tile_contig, d_bits, d_last, ss);
            MG_LAUNCH_CHECK();
            (gen ? k_six_cand<false, true> : k_six_cand<false, false>)<<<cand_grid, 32 * CAND_WARPS, 0, st>>>(
                g->d_packed, nullptr, 0, s->d_tile_base, s->d_cid, g->d_contig_len, g->d_contig_base, s->d_cs, s->d_m, s->d_tile_contig,
                s->n_tiles, d_bits, d_last, min_aa, s->d_cnt, s->d_hits, s->hit_cap, s->d_hit_count, ss);
            MG_LAUNCH_CHECK();
        }
    } else {
        (gen ? k_six_scan<true> : k_six_scan<false>)<<<(unsigned)s->n_tiles, SIX_THREADS, 0, st>>>(
            g->d_packed, s->d_tile_base, nc, s->d_cid, g->d_contig_len, g->d_contig_base, s->d_cs, s->d_m, s->d_tile_contig, s->n_tiles,
            s->d_look, s->d_carry, min_aa, 2 * g->total_bases, s->d_cnt, s->d_hits, s->hit_cap, s->d_hit_count, ss);
        MG_LAUNCH_CHECK();
    }
    s->scan_tmp_cap = mg_scan_tmp_elems(s->n_tiles * 6) + 2;
    TRY(six_alloc(s, &s->d_scan_tmp, s->scan_tmp_cap));
    TRY(mg_scan_i32(s->d_cnt, s->d_cnt_off, s->n_tiles * 6, s->d_scan_tmp, s->scan_tmp_cap, st));
    MG_CUDA(cudaMemcpyAsync(&s->n_orf, s->d_cnt_off + s->n_tiles * 6, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MG_CUDA(cudaStreamSynchronize(st));
    if (use_two_level && s->n_orf > s->hit_cap) {     // more kept ORFs than the hit list holds: the single-pass scan + dense emit
#undef TRY
        std::vector<int64_t> ids(contig_ids, contig_ids + n_list);
        mg_sixframe_free(g);
        g_six_force_single = true;
        const int rc2 = six_count(g, n_list, ids.data(), min_aa, codon64, orf, n_orf, n_bytes, stream);
        g_six_force_single = false;
        return rc2;
#define TRY(x) do { rc = (x); if (rc) return rc; } while (0)
    }
    if (s->n_orf > 0) {
        TRY(six_alloc(s, &s->d_recs, s->n_orf));
        TRY(six_alloc(s, &s->d_len, s->n_orf));
        TRY(six_alloc(s, &s->d_src, s->n_orf));
        TRY(six_alloc(s, &s->d_aa_off, s->n_orf + 1));
        if (s->n_orf <= s->hit_cap) {
            k_six_place<<<(unsigned)((s->n_orf + 255) / 256), 256, 0, st>>>(s->d_hits, s->n_orf, s->d_tile_base, nc, s->d_cid, g->d_contig_len,
                                                                            g->d_contig_base, s->d_cs, s->d_m, s->d_cnt_off, 2 * g->total_bases,
                                                                            s->d_recs, s->d_len, s->d_src);
        } else {                                     // dense output (tiny min_aa): second pass over the genome
            (gen ? k_six_orfs<true, true> : k_six_orfs<true, false>)<<<(unsigned)s->n_tiles, SIX_THREADS, 0, st>>>(
                g->d_packed, s->d_tile_base, nc, s->d_cid, g->d_contig_len, g->d_contig_base, s->d_cs, s->d_m, s->n_tiles, s->d_carry,
                min_aa, 2 * g->total_bases, nullptr, s->d_cnt_off, s->d_recs, s->d_len, s->d_src, ss);
        }
        MG_LAUNCH_CHECK();
        if (orf) TRY(orf_select(g, s, orf->start64, orf->partial, min_aa));          // the segments -> the ORFs (s->n_orf may drop to 0)
    }
    if (s->n_orf > 0) {
        const int64_t need = mg_scan_tmp_elems(s->n_orf) + 2;
        int64_t *tmp = s->d_scan_tmp;
        if (need > s->scan_tmp_cap) TRY(six_alloc(s, &tmp, need));
        TRY(mg_scan_i32(s->d_len, s->d_aa_off, s->n_orf, tmp, std::max(need, s->scan_tmp_cap), st));
        if (orf) k_orf_fill_off<<<(unsigned)((s->n_orf + 255) / 256), 256, 0, st>>>(s->n_orf, s->d_aa_off, s->d_calls);
        else k_six_fill_off<<<(unsigned)((s->n_orf + 255) / 256), 256, 0, st>>>(s->n_orf, s->d_aa_off, s->d_recs);
        MG_LAUNCH_CHECK();
        MG_CUDA(cudaMemcpyAsync(&s->n_bytes, s->d_aa_off + s->n_orf, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        MG_CUDA(cudaStreamSynchronize(st));
        s->n_aa_tile = (s->n_bytes + AA_TILE - 1) / AA_TILE;
        TRY(six_alloc(s, &s->d_aa_tile, s->n_aa_tile + 1));
        if (s->n_aa_tile > 0) {
            k_six_tiles<<<(unsigned)((s->n_aa_tile + 256) / 256), 256, 0, st>>>(s->d_aa_off, s->n_orf, AA_TILE, s->n_aa_tile, s->d_aa_tile);
            MG_LAUNCH_CHECK();
        }
    }
#undef TRY
    if (n_orf) *n_orf = s->n_orf;
    if (n_bytes) *n_bytes = s->n_bytes;
    return MG_OK;
}

// contigs given as a LIST (any order, e.g. the LPT share of one GPU): ORFs come out contig by contig in list order
extern "C" int mg_sixframe_count_list_table(mg_genome *g, int64_t n_list, const int64_t *contig_ids, int64_t min_aa,
                                            const uint8_t *codon64, int64_t *n_orf, int64_t *n_bytes, void *stream) {
    const int rc = six_validate(g, n_list, contig_ids, min_aa, codon64);
    if (rc) return rc;
    return six_count(g, n_list, contig_ids, min_aa, codon64, nullptr, n_orf, n_bytes, stream);
}

extern "C" int mg_orfcall_count(mg_genome *g, int64_t n_list, const int64_t *contig_ids, int64_t min_aa, const uint8_t *codon64,
                                const uint8_t *start64, int partial, int64_t *n_orf, int64_t *n_bytes, void *stream) {
    const int rc = six_validate(g, n_list, contig_ids, min_aa, codon64);
    if (rc) return rc;
    uint8_t atg[64] = {0};
    atg[14] = 1;                                                // ATG: 16*0 + 4*3 + 2 (A=0 C=1 G=2 T=3)
    if (!start64) start64 = atg;
    uint8_t std64[64];
    if (!codon64) {                                             // the standard code's stops: TAA TAG TGA
        memset(std64, 'X', 64);
        std64[48] = std64[50] = std64[56] = '*';
    }
    const uint8_t *stops = codon64 ? codon64 : std64;
    bool any = false;
    for (int c = 0; c < 64; c++) {
        if (!start64[c]) continue;
        any = true;
        if (stops[c] == '*') {
            mg_set_error("start codon %c%c%c is a stop codon of this genetic code", "ACGT"[c >> 4], "ACGT"[(c >> 2) & 3], "ACGT"[c & 3]);
            return MG_EINVAL;
        }
    }
    MG_REQUIRE(any, "start64 flags no start codon");
    const OrfSel sel = {start64, partial != 0};
    return six_count(g, n_list, contig_ids, min_aa, codon64, &sel, n_orf, n_bytes, stream);
}

extern "C" int mg_sixframe_count_list(mg_genome *g, int64_t n_list, const int64_t *contig_ids, int64_t min_aa, int64_t *n_orf,
                                      int64_t *n_bytes, void *stream) {
    return mg_sixframe_count_list_table(g, n_list, contig_ids, min_aa, nullptr, n_orf, n_bytes, stream);
}

extern "C" int mg_sixframe_count_table(mg_genome *g, int64_t contig_lo, int64_t contig_hi, int64_t min_aa, const uint8_t *codon64,
                                       int64_t *n_orf, int64_t *n_bytes, void *stream) {
    MG_REQUIRE(g != nullptr, "genome handle is NULL");
    MG_REQUIRE(contig_lo >= 0 && contig_lo <= contig_hi && contig_hi <= g->n_contigs, "contig range out of bounds");
    std::vector<int64_t> ids(contig_hi - contig_lo);
    for (int64_t i = 0; i < (int64_t)ids.size(); i++) ids[i] = contig_lo + i;
    return mg_sixframe_count_list_table(g, (int64_t)ids.size(), ids.data(), min_aa, codon64, n_orf, n_bytes, stream);
}

extern "C" int mg_sixframe_count(mg_genome *g, int64_t contig_lo, int64_t contig_hi, int64_t min_aa, int64_t *n_orf,
                                 int64_t *n_bytes, void *stream) {
    return mg_sixframe_count_table(g, contig_lo, contig_hi, min_aa, nullptr, n_orf, n_bytes, stream);
}

// residues of the counted ORFs into out_dev (16-byte aligned); ORF calls get their first residue set to M
static int six_residues(mg_genome *g, uint8_t *out_dev, cudaStream_t st) {
    mg_sixframe_state *s = g->six;
    if (!out_dev || s->n_bytes <= 0) return MG_OK;
    MG_REQUIRE(((uintptr_t)out_dev & 15) == 0, "aa_out_dev must be 16-byte aligned");
    k_six_aa<<<(unsigned)s->n_aa_tile, AA_THREADS, 0, st>>>(g->d_packed, s->d_aa_off, s->d_src, s->n_orf, s->d_aa_tile, s->n_bytes,
                                                            s->d_aa4096 ? s->d_aa4096 : g->d_aa4096, out_dev);
    MG_LAUNCH_CHECK();
    if (s->orfcall) {
        k_orf_first_m<<<(unsigned)((s->n_orf + 255) / 256), 256, 0, st>>>(s->n_orf, s->d_aa_off, out_dev);
        MG_LAUNCH_CHECK();
    }
    return MG_OK;
}

// MG_ESTATE unless the preceding count is of this kind and the genome is still the one it scanned
static int six_check_counted(mg_genome *g, bool orfcall) {
    MG_REQUIRE(g != nullptr, "genome handle is NULL");
    if (!g->six || !g->six->counted || g->six->orfcall != orfcall) {
        mg_set_error(orfcall ? "mg_orfcall_count has not been called" : "mg_sixframe_count has not been called");
        return MG_ESTATE;
    }
    if (g->six->generation != g->generation) {
        mg_set_error("the genome changed (pack, finalize or mask) since %s: count again",
                     orfcall ? "mg_orfcall_count" : "mg_sixframe_count");
        return MG_ESTATE;
    }
    return MG_OK;
}

static int six_emit_device(mg_genome *g, bool orfcall, uint8_t *aa_out_dev, void *recs_dev, void *stream) {
    const int rc0 = six_check_counted(g, orfcall);
    if (rc0) return rc0;
    MG_CUDA(cudaSetDevice(g->device));
    cudaStream_t st = (cudaStream_t)stream;
    mg_sixframe_state *s = g->six;
    const int rc = six_residues(g, aa_out_dev, st);
    if (rc) return rc;
    if (recs_dev && s->n_orf > 0)
        MG_CUDA(cudaMemcpyAsync(recs_dev, orfcall ? (void *)s->d_calls : (void *)s->d_recs,
                                s->n_orf * (orfcall ? sizeof(mg_orfcall) : sizeof(mg_orf)), cudaMemcpyDeviceToDevice, st));
    return MG_OK;
}

static int six_emit_host(mg_genome *g, bool orfcall, uint8_t *aa_out_host, void *recs_host, void *stream) {
    const int rc0 = six_check_counted(g, orfcall);
    if (rc0) return rc0;
    MG_CUDA(cudaSetDevice(g->device));
    cudaStream_t st = (cudaStream_t)stream;
    mg_sixframe_state *s = g->six;
    if (aa_out_host && s->n_bytes > 0) {
        const int64_t need = (s->n_bytes + 15) / 16 * 16;
        if (s->aa_cap < need) {
            if (s->d_aa) MG_CUDA(cudaFree(s->d_aa));
            s->d_aa = nullptr;
            s->aa_cap = 0;
            MG_CUDA(cudaMalloc(&s->d_aa, need));
            s->aa_cap = need;
        }
        int rc = six_residues(g, s->d_aa, st);
        if (rc) return rc;
        MG_CUDA(cudaMemcpyAsync(aa_out_host, s->d_aa, s->n_bytes, cudaMemcpyDeviceToHost, st));
    }
    if (recs_host && s->n_orf > 0)
        MG_CUDA(cudaMemcpyAsync(recs_host, orfcall ? (void *)s->d_calls : (void *)s->d_recs,
                                s->n_orf * (orfcall ? sizeof(mg_orfcall) : sizeof(mg_orf)), cudaMemcpyDeviceToHost, st));
    MG_CUDA(cudaStreamSynchronize(st));
    return MG_OK;
}

extern "C" int mg_sixframe_emit_device(mg_genome *g, uint8_t *aa_out_dev, mg_orf *recs_dev, void *stream) {
    return six_emit_device(g, false, aa_out_dev, recs_dev, stream);
}

extern "C" int mg_sixframe_emit(mg_genome *g, uint8_t *aa_out_host, mg_orf *recs_host, void *stream) {
    return six_emit_host(g, false, aa_out_host, recs_host, stream);
}

extern "C" int mg_orfcall_emit_device(mg_genome *g, uint8_t *aa_out_dev, mg_orfcall *recs_dev, void *stream) {
    return six_emit_device(g, true, aa_out_dev, recs_dev, stream);
}

extern "C" int mg_orfcall_emit(mg_genome *g, uint8_t *aa_out_host, mg_orfcall *recs_host, void *stream) {
    return six_emit_host(g, true, aa_out_host, recs_host, stream);
}
