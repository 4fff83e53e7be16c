// mg_common.cuh -- shared host/device definitions of libmagot_b200 (sm_100a only).
//
// Genome layout in HBM (one allocation per genome handle):
//   packed[]  : uint32 words, 8 bases per word, base g lives in bits [4*(g&7), 4*(g&7)+4) of word g>>3
//               nibble codes: 0-3 = A C G T, 4-7 = a c g t, 8 = N, 9 = n, 10 = '-', 11-14 = R Y K M,
//               15 = exception (exact byte kept in the sorted side list exc_pos[] / exc_byte[]).
//               complement of codes 0..7 is code ^ 3 (case bit 2 is preserved), which is what makes the
//               reverse complement (genome.py:784-793) three register ops per 8 bases.
//   contigs are laid back to back in one global base index space; contig c starts at contig_base[c],
//   a multiple of 32 bases (16 bytes); index 0..63 is front padding so that a window that
//   starts a little before the first base of the genome can still be loaded with non-negative addresses.
//   TWO PLANES: indices [0, T) hold the forward strand, indices [T, 2T) hold the reverse complement of
//   the whole index space (base g of the forward plane is base 2T-1-g of the reverse plane, complemented
//   in code space, codes 11..15 already turned into 'n' as Sequence.reverse_compliment does).  A '-' strand
//   interval is therefore a plain FORWARD read of the second plane: the kernels never branch on strand
//   and never reverse in registers.  This doubles the resident footprint to 1 B/base (3.1 GB for a human
//   genome on a 180 GB part) and leaves the HBM traffic per spliced base at 0.5 B; the round-1 ncu profile
//   showed the emit kernels issue-bound, not bandwidth-bound, which is what this trade buys back.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <string>
#include <vector>
#include "../../include/magot_b200.h"

#define MG_FRONT_PAD 64            // bases of padding before contig 0 (K3 may start a 48-nibble window 45 bases early)
#define MG_TAIL_WORDS 8            // readable slack words after the last contig
#define MG_CODE_EXC 15u

// ---- host-side error plumbing -----------------------------------------------------------------
void mg_set_error(const char *fmt, ...);
extern std::atomic<int64_t> g_mg_launches;        // kernels launched by this library (any host thread)
#define MG_COUNT_LAUNCH() (++g_mg_launches)

#define MG_CUDA(call)                                                                             \
    do {                                                                                          \
        cudaError_t _e = (call);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            mg_set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return MG_ECUDA;                                                                      \
        }                                                                                         \
    } while (0)

#define MG_LAUNCH_CHECK()                                                                         \
    do {                                                                                          \
        MG_COUNT_LAUNCH();                                                                        \
        cudaError_t _e = cudaGetLastError();                                                      \
        if (_e != cudaSuccess) {                                                                  \
            mg_set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return MG_ECUDA;                                                                      \
        }                                                                                         \
    } while (0)

#define MG_REQUIRE(cond, msg)                                                                     \
    do {                                                                                          \
        if (!(cond)) {                                                                            \
            mg_set_error("%s (%s:%d)", msg, __FILE__, __LINE__);                                  \
            return MG_EINVAL;                                                                     \
        }                                                                                         \
    } while (0)

// ---- handles -------------------------------------------------------------------------------------
struct mg_sixframe_state;

struct mg_genome {
    int device = 0;
    int64_t n_contigs = 0;
    int64_t total_bases = 0;                  // T: padded global index space of ONE plane (incl. front pad)
    std::vector<int64_t> h_contig_len, h_contig_base;
    uint32_t *d_packed = nullptr;             // 2*total_bases/8 + MG_TAIL_WORDS words (forward plane, reverse plane)
    int64_t *d_contig_len = nullptr, *d_contig_base = nullptr;
    // exceptions, unsorted while packing (device), sorted after finalize
    int64_t *d_exc_pos = nullptr;
    uint8_t *d_exc_byte = nullptr;
    int64_t exc_cap = 0;
    int64_t n_exc = 0;
    unsigned long long *d_exc_count = nullptr;
    std::vector<int64_t> h_exc_pos;           // collected per chunk
    std::vector<uint8_t> h_exc_byte;
    bool finalized = false;
    uint64_t generation = 0;                  // bumped by every call that can change the bases (pack*, finalize, mask): a count or
                                              // plan prepared at another generation cannot be emitted (MG_ESTATE)
    uint8_t *d_stage = nullptr;               // H2D staging for pack / fetch
    int64_t stage_cap = 0;
    uint8_t *d_raw = nullptr;                 // raw FASTA body chunk (mg_genome_pack_fasta)
    unsigned long long *d_strip_tmp = nullptr;    // look-back words of k_fasta_strip + the kept-byte total
    int64_t raw_cap = 0;
    uint8_t *h_pin = nullptr;                 // pinned bounce buffer
    int64_t pin_cap = 0;
    uint8_t *d_aa4096 = nullptr;              // 4096-entry nibble-triplet -> amino acid table
    uint8_t *d_aa4096h = nullptr;             // the same, entry of codon c stored at mg_aa_slot(c) (shared-memory friendly)
    uint32_t *d_stops = nullptr;              // stop-codon index (K4): one bit per base and strand, [0, stop_words) plus, [stop_words, 2 stop_words) minus
    int64_t stop_words = 0;
    bool stops_valid = false;                 // false after pack / mask: rebuilt by the next ORF scan
    uint32_t *d_stops_alt = nullptr;          // the same for ONE other stop set (a non-standard genetic code), same layout
    uint64_t stops_alt_key = 0;               // its stop codons: bit 16*b0 + 4*b1 + b2 (A=0 C=1 G=2 T=3)
    bool stops_alt_valid = false;             // false after pack / mask, like stops_valid
    mg_sixframe_state *six = nullptr;
    int64_t device_bytes = 0;
};

struct mg_plan {
    mg_genome *g = nullptr;
    int device = 0;
    int64_t n_rec = 0, n_seg = 0, n_piece = 0, n_lit = 0;
    // inputs (device copies)
    int64_t *d_rec_seg_off = nullptr;         // [n_rec+1]
    int32_t *d_seg_contig = nullptr;
    int64_t *d_seg_start = nullptr, *d_seg_end = nullptr;
    int8_t *d_seg_strand = nullptr;
    int64_t *d_rec_lit_off = nullptr;
    int32_t *d_rec_pre = nullptr, *d_rec_suf = nullptr;
    int8_t *d_rec_phase = nullptr;
    uint8_t *d_lit = nullptr;
    // derived (device)
    int64_t *d_blk_r0 = nullptr;              // [n_piece/256] record owning the first piece of each 256-piece block
    int64_t *d_piece_src = nullptr;           // [n_piece]  src | kind<<62
    int64_t *d_piece_off = nullptr;           // [n_piece+1] exclusive prefix = offsets in the nucleotide text
    int64_t *d_prot_off = nullptr;            // [n_rec+1]
    int32_t *d_rec_aa = nullptr;              // [n_rec] amino acids, -1 = reference returns None
    int8_t *d_rec_skip = nullptr;             // [n_rec] spliced bases skipped before the first codon (0..3)
    int64_t *d_nuc_tile = nullptr;            // first piece of each nucleotide tile
    int64_t *d_prot_tile = nullptr;           // first record of each protein tile
    int64_t n_nuc_tile = 0, n_prot_tile = 0;
    int32_t *d_blk1k = nullptr;               // first piece of every 1 KB block of the nucleotide text (+ sentinel), for k_emit_nuc_stream
    int64_t blk1k_cap = 0;                    // entries the table can take (from the host-side upper bound of the text size)
    bool blk1k_ready = false;                 // filled by the last prepare (only when the streaming K2 variant was selected then)
    int64_t max_seg_per_rec = 0;             // longest record (segments): k_plan_rec walks a record with one thread
    int64_t nuc_upper = 0;                    // host-side upper bound of the nucleotide text size: sum(max(0, end-start+1)) + framing
    int64_t *d_tile_buf = nullptr;
    int64_t tile_cap = 0;
    cudaStream_t last_stream = 0;             // frees are ordered after the last use on this stream
    int64_t *d_scan_tmp = nullptr;            // block sums for scans
    int64_t scan_tmp_cap = 0;
    int64_t nuc_total = -1, prot_total = -1;      // text sizes on the host; with mg_plan_prepare_async: the caller's upper bounds
    int64_t prot_cap = 0;                         // the protein capacity given to mg_plan_prepare_async
    int64_t *d_totals = nullptr;                  // [2] the same on the device (written by the plan kernels)
    bool totals_known = false;                    // false between mg_plan_prepare_async and mg_plan_totals
    int prot_flags = 0;
    bool prepared = false;
    uint64_t generation = 0;                      // g->generation at the last prepare: K1 read the bases then, the emits read them again
    bool prot_ready = false;                      // false between mg_plan_prepare_async(MG_PROT_DEFER) and mg_plan_prepare_prot_async
    unsigned long long *rec_tmp = nullptr;        // look-back words / tile table of the deferred record pass
    int64_t rec_tmp_words = 0;
    int64_t *rec_tile = nullptr;
    uint32_t *d_order = nullptr;              // rank -> (job, tile) of mg_emit_products_device launches led by this plan
    int64_t order_cap = 0;
    uint8_t *d_out = nullptr;                 // library-owned output buffer for *_host emits
    int64_t out_cap = 0;
    uint8_t *d_aa8192 = nullptr;              // the plan's own translation tables (mg_plan_set_codon_table): plain | mg_aa_slot order
    bool own_code = false;                    // true: K3 / K23 / the one-launch emit read d_aa8192 instead of the genome's tables
    uint64_t stop_mask = 0;                   // stop codons of the plan's code, bit 16*b0 + 4*b1 + b2 (mg_plan_check)
    // the caller's segment table as given to mg_plan_create (mg_plan_check reports junctions per caller segment); the same
    // pointers as the plan's own table unless a segment of 2^31 bases or more was split into chunks
    int64_t n_cseg = 0;
    int64_t *d_crec_seg_off = nullptr;
    int32_t *d_cseg_contig = nullptr;
    int64_t *d_cseg_start = nullptr, *d_cseg_end = nullptr;
    int8_t *d_cseg_strand = nullptr;
    mg_cds_check *d_chk = nullptr;            // device outputs of the host-buffer mg_plan_check
    uint32_t *d_chk_counts = nullptr;
    int8_t *d_chk_junction = nullptr;
    mg_cds_pred *d_pred = nullptr;            // device outputs of the host-buffer mg_plan_predict_cds
    mg_cds_seg *d_pred_seg = nullptr;
    std::vector<void *> owned;                // everything to free
};

#define MG_STD_STOPS ((1ull << 48) | (1ull << 50) | (1ull << 56))   // TAA TAG TGA, bit 16*b0 + 4*b1 + b2 (A=0 C=1 G=2 T=3)

#define MG_KIND_FWD 0ull
#define MG_KIND_RC 1ull
#define MG_KIND_LIT 2ull
#define MG_KIND_SHIFT 62
#define MG_SRC_MASK ((1ull << MG_KIND_SHIFT) - 1ull)

#ifndef MG_NUC_TILE
#define MG_NUC_TILE 32768          // bytes of nucleotide text per CTA tile
#endif
#ifndef MG_PROT_TILE
#define MG_PROT_TILE 16384         // bytes of protein text per CTA tile
#endif

// internal cross-file helpers
void build_aa4096(uint8_t *t, const uint8_t *codon64);   // nibble-triplet -> residue table from a codon64 table (NULL = standard code)
int mg_plan_check_prepared(const mg_plan *p);         // MG_ESTATE unless p was prepared and its genome has not changed since
int mg_refuse_growth_in_capture(cudaStream_t st, const char *what);   // MG_ESTATE when st is being captured (a buffer would have to grow)
int mg_start_mask(const mg_plan *p, const uint8_t *start64, uint64_t *mask);   // start64 flags (NULL = ATG) as a bit set, checked against the plan's stops
int mg_scan_i32(const int32_t *d_in, int64_t *d_out, int64_t n, int64_t *d_tmp, int64_t tmp_cap, cudaStream_t st);
int64_t mg_scan_tmp_elems(int64_t n);
int mg_ensure_stage(mg_genome *g, int64_t bytes);
int mg_ensure_pin(mg_genome *g, int64_t bytes);
void mg_parallel_copy(const uint8_t *src, uint8_t *dst, int64_t n);   // memcpy on up to 8 host threads (pageable <-> page-locked staging)
int mg_emit_mode();                                   // K2 variant, env MAGOT_EMIT: 0 = ldg (mg_emit.cu, default: the fastest), 1 = tma (mg_emit_tma.cu), 2 = stream (mg_emit_stream.cu)
int mg_launch_nuc_tma(mg_plan *p, uint8_t *out_dev, cudaStream_t st);
int mg_launch_nuc_stream(mg_plan *p, uint8_t *out_dev, cudaStream_t st);
void mg_set_fuse(int v);                              // mg_tune("fuse", 0/1): K23 as one fused launch (1, default) or K2 + K3
void mg_set_multi_lag(int ppm);                       // lag between the jobs of mg_emit_products_device (mg_tune("multi_lag", ppm))

#ifdef __CUDACC__
// ---- device primitives -----------------------------------------------------------------------------

// 16 consecutive nibbles starting at global base index g (g >= 0), base g in bits 0..3.
__device__ __forceinline__ uint64_t mg_ld_nib16(const uint32_t *__restrict__ pk, int64_t g) {
    const uint32_t *p = pk + (g >> 3);
    const uint32_t sh = ((uint32_t)g & 7u) << 2;
    const uint32_t w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2);
    const uint32_t lo = __funnelshift_r(w0, w1, sh);
    const uint32_t hi = __funnelshift_r(w1, w2, sh);
    return ((uint64_t)hi << 32) | lo;
}

__device__ __forceinline__ uint32_t mg_rev_nib32(uint32_t x) {
    x = __byte_perm(x, 0, 0x0123);
    return ((x & 0x0F0F0F0Fu) << 4) | ((x >> 4) & 0x0F0F0F0Fu);
}

// complement in code space (genome.py:787): 0..7 -> ^3, 8/9/10 (N n -) unchanged, 11..15 -> 9 ('n')
__device__ __forceinline__ uint32_t mg_comp_nib32(uint32_t x) {
    const uint32_t b3 = (x >> 3) & 0x11111111u;
    if (b3 == 0) return x ^ 0x33333333u;
    const uint32_t m = b3 * 15u;
    const uint32_t f = b3 & ((x >> 2) | ((x >> 1) & x));
    const uint32_t y = x ^ (0x33333333u & ~m);
    return (y & ~(f * 15u)) | (f * 9u);
}

// reverse complement of 16 nibbles: out nibble j = comp(in nibble 15-j)
__device__ __forceinline__ uint64_t mg_rc_nib16(uint64_t v) {
    const uint32_t lo = mg_comp_nib32(mg_rev_nib32((uint32_t)(v >> 32)));
    const uint32_t hi = mg_comp_nib32(mg_rev_nib32((uint32_t)v));
    return ((uint64_t)hi << 32) | lo;
}

// 8 nibbles -> 8 ASCII bytes.  Code 15 decodes to '?' and must be patched by the caller.
// Branch-free: two 8-entry byte tables per half (PRMT), chosen per byte by bit 3 of the nibble.  The byte mask for
// "bit 3 set" is one PRMT in sign-replicate mode: for the 16 bits n3 n2 n1 n0 of four nibbles, bit 3 of n1/n3 is the
// sign bit of byte 0/1 of x, and bit 3 of n0/n2 is the sign bit of byte 0/1 of x << 4.
__device__ __forceinline__ void mg_decode8(uint32_t x, uint32_t &o0, uint32_t &o1) {
    const uint32_t LA = 0x54474341u;  // "ACGT"
    const uint32_t LB = 0x74676361u;  // "acgt"
    const uint32_t LC = 0x522D6E4Eu;  // "Nn-R"
    const uint32_t LD = 0x3F4D4B59u;  // "YKM?"
#ifdef MG_DECODE_BRANCHY
    const uint32_t s = x & 0x77777777u;
    o0 = __byte_perm(LA, LB, s & 0xFFFFu);
    o1 = __byte_perm(LA, LB, s >> 16);
    const uint32_t h = x & 0x88888888u;
    if (h) {
        const uint32_t h0 = __byte_perm(LC, LD, s & 0xFFFFu);
        const uint32_t h1 = __byte_perm(LC, LD, s >> 16);
        uint32_t t = h & 0xFFFFu;
        uint32_t m0 = ((t & 0x8u) << 4) | ((t & 0x80u) << 8) | ((t & 0x800u) << 12) | ((t & 0x8000u) << 16);
        t = h >> 16;
        uint32_t m1 = ((t & 0x8u) << 4) | ((t & 0x80u) << 8) | ((t & 0x800u) << 12) | ((t & 0x8000u) << 16);
        m0 = (m0 >> 7) * 0xFFu;             // bit 7 of each byte -> 0xFF / 0x00 byte mask
        m1 = (m1 >> 7) * 0xFFu;
        o0 = (o0 & ~m0) | (h0 & m0);
        o1 = (o1 & ~m1) | (h1 & m1);
    }
#else
    const uint32_t s = x & 0x77777777u, s1 = s >> 16;
    const uint32_t x4 = x << 4;
    uint32_t m0, m1;                                      // (__byte_perm drops selector bit 3, the sign-replicate flag)
    asm("prmt.b32 %0, %1, %2, 0xD9C8;" : "=r"(m0) : "r"(x4), "r"(x));   // sign(x4.b0), sign(x.b0), sign(x4.b1), sign(x.b1)
    asm("prmt.b32 %0, %1, %2, 0xFBEA;" : "=r"(m1) : "r"(x4), "r"(x));   // same for bytes 2, 3
    const uint32_t a0 = __byte_perm(LA, LB, s), a1 = __byte_perm(LA, LB, s1);
    const uint32_t h0 = __byte_perm(LC, LD, s), h1 = __byte_perm(LC, LD, s1);
    o0 = (a0 & ~m0) | (h0 & m0);
    o1 = (a1 & ~m1) | (h1 & m1);
#endif
}

// Slot of the 12-bit codon c (three nibbles, first base lowest) in the shared-memory copy of the translation table.
// With the plain index, the 4-byte word -- hence the bank -- of a valid codon is chosen by the first base's case bit and the
// second base alone: 32 lanes hit 4 banks (measured 3.98 wavefronts per lookup).  XOR-ing the third base into index bits
// 2-3 makes the bank (base3, base2, case) and leaves the first base as the byte inside the word: lanes that share a bank
// now share the word, so a lookup is one wavefront unless the case changes inside a codon.  A bijection on 12 bits.
__host__ __device__ __forceinline__ uint32_t mg_aa_slot(uint32_t c) {
    return (c ^ ((c >> 6) & 0xCu)) & 0xFFFu;
}

// ASCII -> nibble code (pack side)
__device__ __forceinline__ uint32_t mg_encode(uint8_t c) {
    switch (c) {
    case 'A': return 0; case 'C': return 1; case 'G': return 2; case 'T': return 3;
    case 'a': return 4; case 'c': return 5; case 'g': return 6; case 't': return 7;
    case 'N': return 8; case 'n': return 9; case '-': return 10;
    case 'R': return 11; case 'Y': return 12; case 'K': return 13; case 'M': return 14;
    default: return MG_CODE_EXC;
    }
}

// exact byte of an exception position (binary search in the sorted side list)
__device__ __forceinline__ uint8_t mg_exc_byte(const int64_t *__restrict__ pos, const uint8_t *__restrict__ byt,
                                               int64_t n, int64_t g) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(pos + mid) < g) lo = mid + 1; else hi = mid;
    }
    return (lo < n && __ldg(pos + lo) == g) ? __ldg(byt + lo) : (uint8_t)'?';
}

// largest i in [lo, hi) with a[i] <= x, given a[lo] <= x  (upper_bound - 1)
__device__ __forceinline__ int64_t mg_search_le(const int64_t *__restrict__ a, int64_t lo, int64_t hi, int64_t x) {
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= x) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ void mg_st16(uint8_t *p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
#endif  // __CUDACC__
