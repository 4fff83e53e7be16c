// mg_predict.cu -- CDS prediction of a prepared plan (mg_plan_predict_cds*): the longest ORF of every record's spliced payload in
// its three frames, mapped back to the caller's segments.  Semantics: include/magot_b200.h.
//
// Two launches on one stream, no host round trip:
//   k_predict_scan  one warp per record walks the payload 512 positions per step.  Lane l owns positions [16l, 16l + 16) of the
//                   step: it builds the 18 nibbles they need from the record's pieces with K3's window (one one-sided mask per
//                   piece), turns them into three bit planes (base bit 0, base bit 1, outside A/C/G/T) and gets the 16 stop and
//                   start flags from logic on the planes, one AND chain per codon of the set (no look-up per position).  Per
//                   frame, "is there a stop" and "the first start after the last stop" are carried across lanes by one warp
//                   scan and across steps in registers; each lane then closes the ORFs of its own stops and keeps its best
//                   (n_aa, -lo) key.  One warp max at the end, then the open 3' ends and the two codons of the winner;
//   k_predict_map   one thread per record walks its caller segments (the table given to mg_plan_create, not the plan's
//                   chunks of long segments), clamps them as the plan does and writes each one's share of the ORF.
// Every genome and payload index is 64-bit.
#include <algorithm>
#include <climits>
#include "mg_common.cuh"
#include "mg_gather.cuh"
#include "mg_emit_common.cuh"

#define PRD_THREADS 256
#define PRD_STEP 512                                   // payload positions per warp step (16 a lane)
#define PRD_NONE 0x3FFu                                // scan field: no start (larger than every step position)
#define PRD_STOP 0x400u                                // scan field: the range holds a stop
#define PRD_IDENT (0x3FFull | (0x3FFull << 16) | (0x3FFull << 32))
#define PRD_LO_MASK ((1ull << 33) - 1ull)              // a payload is shorter than 2^33 bases (3 * (2^31 - 1) + 2)

static_assert(sizeof(mg_cds_pred) == 32, "mg_cds_pred layout (include/magot_b200.h)");
static_assert(sizeof(mg_cds_seg) == 24, "mg_cds_seg layout (include/magot_b200.h)");

struct PrdArgs {
    const uint32_t *packed;
    const int64_t *piece_off, *piece_src, *rec_seg_off;
    int64_t n_rec, min_aa;
    uint64_t stop_mask, start_mask;
    int flags;
    mg_cds_pred *rec;
};

// bit s of each of the 8 nibbles of x, as 8 bits
__device__ __forceinline__ uint32_t prd_plane8(uint32_t x, int s) {
    uint32_t t = (x >> s) & 0x11111111u;
    t = (t | (t >> 3)) & 0x03030303u;
    t = (t | (t >> 6)) & 0x000F000Fu;
    return (t | (t >> 12)) & 0xFFu;
}

// positions whose base is b (A=0 C=1 G=2 T=3), from the planes of base bit 0, base bit 1 and "inside A/C/G/T"
__device__ __forceinline__ uint32_t prd_base(uint32_t b0, uint32_t b1, uint32_t ok, uint32_t b) {
    return ok & ((b & 2u) ? b1 : ~b1) & ((b & 1u) ? b0 : ~b0);
}

// the 16 codon starts of an 18-nibble window whose codon is in `set` (bit 16*b0 + 4*b1 + b2); `set` is warp-uniform
__device__ __forceinline__ uint32_t prd_codons(uint64_t set, uint32_t b0, uint32_t b1, uint32_t ok) {
    uint32_t m = 0;
    while (set) {
        const uint32_t c = (uint32_t)(__ffsll((long long)set) - 1);
        set &= set - 1;
        m |= prd_base(b0, b1, ok, c >> 4) & (prd_base(b0, b1, ok, (c >> 2) & 3u) >> 1) & (prd_base(b0, b1, ok, c & 3u) >> 2);
    }
    return m & 0xFFFFu;
}

// scan operator per frame (16-bit field: PRD_STOP | step position of a start): `a` is the earlier range, `b` the later one.
// A range maps the open start o it receives to: its first start after its last stop if it holds a stop, else o when there is
// one, else its first start.
__device__ __forceinline__ uint64_t prd_combine(uint64_t a, uint64_t b) {
    uint64_t r = 0;
#pragma unroll
    for (int f = 0; f < 3; f++) {
        const uint32_t fa = (uint32_t)(a >> (16 * f)) & 0x7FFu, fb = (uint32_t)(b >> (16 * f)) & 0x7FFu;
        const uint32_t fr = (fb & PRD_STOP) ? fb : ((fa & PRD_STOP) | min(fa & PRD_NONE, fb & PRD_NONE));
        r |= (uint64_t)fr << (16 * f);
    }
    return r;
}

// the open start (payload position, -1 = none) after a range with scan field `fld` at step base B, given the open start `o` before
__device__ __forceinline__ int64_t prd_apply(uint32_t fld, int64_t B, int64_t o) {
    const int64_t v = (fld & PRD_NONE) == PRD_NONE ? -1 : B + (int64_t)(fld & PRD_NONE);
    return (fld & PRD_STOP) ? v : (o >= 0 ? o : v);
}

// selection key: more residues first, then the smaller start
__device__ __forceinline__ unsigned long long prd_key(int64_t naa, int64_t lo) {
    return ((unsigned long long)naa << 33) | (PRD_LO_MASK - (unsigned long long)lo);
}

__device__ __forceinline__ uint32_t prd_codon_index(uint32_t c12) {
    if (c12 & 0x888u) return 0xFFu;
    return ((c12 & 3u) << 4) | (((c12 >> 4) & 3u) << 2) | ((c12 >> 8) & 3u);
}

// codon at payload position i of the record whose payload starts in piece f0 + 1 at text offset ns
__device__ __noinline__ uint32_t prd_codon_at(const PrdArgs &a, int64_t f0, int64_t f1, int64_t ns, int64_t i) {
    const int64_t S = ns + i;
    const int64_t j = mg_search_le(a.piece_off, f0 + 1, f1 - 1, S);
    uint64_t acc[3];
    mg_gather_nib(a.packed, a.piece_off, a.piece_src, j, S, 3, acc);
    return prd_codon_index((uint32_t)acc[0] & 0xFFFu);
}

__global__ void __launch_bounds__(PRD_THREADS) k_predict_scan(const __grid_constant__ PrdArgs a) {
    const int64_t r = (blockIdx.x * (int64_t)PRD_THREADS + threadIdx.x) >> 5;
    if (r >= a.n_rec) return;
    const int lane = threadIdx.x & 31;
    const int64_t f0 = __ldg(a.rec_seg_off + r) + 2 * r, f1 = __ldg(a.rec_seg_off + r + 1) + 2 * (r + 1);
    const int64_t ns = __ldg(a.piece_off + f0 + 1), n = __ldg(a.piece_off + f1 - 1) - ns;
    int64_t carry[3];                                  // open start of each frame before the step (-1 = none); warp-uniform
#pragma unroll
    for (int f = 0; f < 3; f++) carry[f] = (a.flags & MG_PRED_5PARTIAL) && f + 3 <= n ? f : -1;
    unsigned long long best = 0;                       // (n_aa << 33) | (2^33 - 1 - lo) of the lane's best ORF with a stop
    int64_t jw = f0 + 1;                               // a piece at or before every window of the step
    int bm3 = 0;                                       // B mod 3
    const int lm3 = lane % 3;                          // 16 * lane mod 3
#pragma unroll 1
    for (int64_t B = 0; B + 2 < n; B += PRD_STEP, bm3 = (bm3 + PRD_STEP) % 3) {
        const int64_t p = B + 16 * lane;
        const int64_t nv64 = n - 2 - p;                // codon starts of the lane: k < nv
        const int nv = (int)max(min(nv64, (int64_t)16), (int64_t)0);
        uint32_t stop16 = 0, start16 = 0;
        int64_t j = jw;
        if (nv > 0) {
            const int64_t P = ns + p;
            j = mg_search_le(a.piece_off, jw, f1 - 1, P);
            uint32_t w[3] = {0, 0, 0};
#pragma unroll 1
            for (int64_t q = j; q < f1 - 1; q++) {
                const int64_t o0 = __ldg(a.piece_off + q);
                if (o0 >= P + 18) break;
                const int64_t o1 = __ldg(a.piece_off + q + 1);
                if (o1 <= o0) continue;                                  // empty piece (clamped-away segment)
                const int c = (int)max(o0 - P, (int64_t)-64);            // window position of the piece's first nibble
                const int64_t g = (int64_t)((uint64_t)__ldg(a.piece_src + q) & MG_SRC_MASK) + (P - o0);
                const uint32_t *pp = a.packed + (g >> 3);
                const uint32_t sh = ((uint32_t)g & 7u) << 2;
                uint32_t v[4];
#pragma unroll
                for (int k = 0; k < 4; k++) v[k] = ld_pk(pp + k);
#pragma unroll
                for (int k = 0; k < 3; k++) {
                    const uint32_t keep = low_nibbles(c - 8 * k);
                    w[k] = (w[k] & keep) | (__funnelshift_r(v[k], v[k + 1], sh) & ~keep);
                }
            }
            const uint32_t b0 = prd_plane8(w[0], 0) | (prd_plane8(w[1], 0) << 8) | (prd_plane8(w[2], 0) << 16);
            const uint32_t b1 = prd_plane8(w[0], 1) | (prd_plane8(w[1], 1) << 8) | (prd_plane8(w[2], 1) << 16);
            const uint32_t ok = ~(prd_plane8(w[0], 3) | (prd_plane8(w[1], 3) << 8) | (prd_plane8(w[2], 3) << 16));
            const uint32_t vmask = nv >= 16 ? 0xFFFFu : ((1u << nv) - 1u);
            stop16 = prd_codons(a.stop_mask, b0, b1, ok) & vmask;
            start16 = prd_codons(a.start_mask, b0, b1, ok) & vmask & ~stop16;
        }
        const int r0 = (bm3 + lm3) % 3;                                  // p mod 3
        uint32_t stp[3], stt[3];
        uint64_t x = 0;
#pragma unroll
        for (int f = 0; f < 3; f++) {
            const int d = (f - r0 + 3) % 3;                              // bits k with (p + k) mod 3 == f
            const uint32_t fm = d == 0 ? 0x9249u : (d == 1 ? 0x2492u : 0x4924u);
            stp[f] = stop16 & fm;
            stt[f] = start16 & fm;
            uint32_t fld;
            if (stp[f]) {
                const int ls = 31 - __clz(stp[f]);
                const uint32_t post = stt[f] & ~((2u << ls) - 1u);
                fld = PRD_STOP | (post ? (uint32_t)(16 * lane + __ffs(post) - 1) : PRD_NONE);
            } else {
                fld = stt[f] ? (uint32_t)(16 * lane + __ffs(stt[f]) - 1) : PRD_NONE;
            }
            x |= (uint64_t)fld << (16 * f);
        }
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint64_t y = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x = prd_combine(y, x);
        }
        uint64_t e = __shfl_up_sync(0xffffffffu, x, 1);
        if (lane == 0) e = PRD_IDENT;
        const uint64_t tot = __shfl_sync(0xffffffffu, x, 31);
#pragma unroll
        for (int f = 0; f < 3; f++) {
            int64_t o = prd_apply((uint32_t)(e >> (16 * f)) & 0x7FFu, B, carry[f]);
            uint32_t s = stp[f], t = stt[f];
            while (s) {                                                  // the ORFs closed by the lane's stops, in order
                const int k = __ffs(s) - 1;
                if (o < 0) {
                    const uint32_t bl = t & ((1u << k) - 1u);
                    if (bl) o = p + __ffs(bl) - 1;
                }
                if (o >= 0) {
                    const int64_t naa = (p + k - o) / 3;
                    if (naa >= a.min_aa) best = max(best, prd_key(naa, o));
                }
                o = -1;
                t &= ~((2u << k) - 1u);
                s &= s - 1;
            }
            carry[f] = prd_apply((uint32_t)(tot >> (16 * f)) & 0x7FFu, B, carry[f]);
        }
        jw = __shfl_sync(0xffffffffu, j, 31);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, d));
    if (lane != 0) return;
    bool stop = best != 0;
    if (a.flags & MG_PRED_3PARTIAL) {                  // the open 3' end of each frame: through its last complete codon
#pragma unroll
        for (int f = 0; f < 3; f++) {
            const int64_t o = carry[f];
            if (o < 0) continue;
            const int64_t hi = f + 3 * ((n - 3 - f) / 3) + 3;
            const int64_t naa = (hi - o) / 3;
            const unsigned long long key = prd_key(naa, o);
            if (naa >= a.min_aa && key > best) { best = key; stop = false; }
        }
    }
    mg_cds_pred out;
    out.n_cds_seg = 0;                                 // k_predict_map counts the segments
    out.pad = 0;
    if (best == 0) {
        out.lo = out.hi = -1;
        out.n_aa = 0;
        out.frame = -1;
        out.type = 0;
        out.start_codon = out.stop_codon = 0xFF;
    } else {
        const int64_t naa = (int64_t)(best >> 33), lo = (int64_t)(PRD_LO_MASK - (best & PRD_LO_MASK));
        const int64_t hi = lo + 3 * naa + (stop ? 3 : 0);
        const uint32_t sc = prd_codon_at(a, f0, f1, ns, lo);
        out.lo = lo;
        out.hi = hi;
        out.n_aa = (int32_t)naa;
        out.frame = (int8_t)(lo % 3);
        out.type = (int8_t)((sc == 0xFFu || !((a.start_mask >> sc) & 1ull) ? 1 : 0) | (stop ? 0 : 2));
        out.start_codon = (uint8_t)sc;
        out.stop_codon = (uint8_t)(stop ? prd_codon_at(a, f0, f1, ns, hi - 3) : 0xFFu);
    }
    a.rec[r] = out;
}

// each caller segment's share of its record's ORF (include/magot_b200.h), and the number of segments the ORF touches
__global__ void __launch_bounds__(256) k_predict_map(int64_t n_rec, const int64_t *__restrict__ rec_seg_off,
                                                     const int32_t *__restrict__ seg_contig, const int64_t *__restrict__ seg_start,
                                                     const int64_t *__restrict__ seg_end, const int8_t *__restrict__ seg_strand,
                                                     const int64_t *__restrict__ contig_len, int64_t n_contigs, mg_cds_pred *rec,
                                                     mg_cds_seg *seg_out) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const int64_t lo = rec[r].lo, hi = rec[r].hi;
    const int64_t e0 = __ldg(rec_seg_off + r), e1 = __ldg(rec_seg_off + r + 1);
    int64_t o = 0;
    int32_t cnt = 0;
    for (int64_t e = e0; e < e1; e++) {
        const int32_t c = __ldg(seg_contig + e);       // contig[start-1:end] with Python slice semantics, as the plan kernels
        int64_t cl = 0, ch = 0;
        if (c >= 0 && c < n_contigs) {
            const int64_t L = __ldg(contig_len + c);
            int64_t i = __ldg(seg_start + e) - 1, j = __ldg(seg_end + e);
            if (i < 0) { i += L; if (i < 0) i = 0; } else if (i > L) i = L;
            if (j < 0) { j += L; if (j < 0) j = 0; } else if (j > L) j = L;
            cl = i;
            ch = j > i ? j : i;
        }
        const int64_t x = max(lo, o), y = min(hi, o + (ch - cl));
        mg_cds_seg s;
        s.lo = s.hi = -1;
        s.phase = -1;
        if (lo >= 0 && x < y) {
            cnt++;
            if (__ldg(seg_strand + e)) { s.lo = ch - (y - o); s.hi = ch - (x - o); }
            else { s.lo = cl + (x - o); s.hi = cl + (y - o); }
            s.phase = (int8_t)((3 - (x - lo) % 3) % 3);
        }
        if (seg_out) {
#pragma unroll
            for (int k = 0; k < 7; k++) s.pad[k] = 0;
            seg_out[e] = s;
        }
        o += ch - cl;
    }
    rec[r].n_cds_seg = cnt;
}

// ---- host API -----------------------------------------------------------------------------------------------

static int pred_args(mg_plan *p, int flags, const uint8_t *start64, uint64_t *start_mask) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    MG_REQUIRE((flags & ~(MG_PRED_5PARTIAL | MG_PRED_3PARTIAL)) == 0, "flags: only MG_PRED_5PARTIAL and MG_PRED_3PARTIAL are accepted");
    if (const int rc = mg_start_mask(p, start64, start_mask)) return rc;
    return mg_plan_check_prepared(p);
}

static int pred_launch(mg_plan *p, int64_t min_aa, uint64_t start_mask, int flags, mg_cds_pred *rec, mg_cds_seg *seg,
                       cudaStream_t st) {
    mg_genome *g = p->g;
    if (p->n_rec == 0) return MG_OK;
    PrdArgs a;
    a.packed = g->d_packed; a.piece_off = p->d_piece_off; a.piece_src = p->d_piece_src; a.rec_seg_off = p->d_rec_seg_off;
    a.n_rec = p->n_rec;
    a.min_aa = std::min(std::max(min_aa, (int64_t)1), (int64_t)1 << 32);      // n_aa is an int32: anything above never passes
    a.stop_mask = p->stop_mask; a.start_mask = start_mask; a.flags = flags; a.rec = rec;
    const int64_t blocks = (p->n_rec + PRD_THREADS / 32 - 1) / (PRD_THREADS / 32);
    k_predict_scan<<<(unsigned)blocks, PRD_THREADS, 0, st>>>(a);
    MG_LAUNCH_CHECK();
    k_predict_map<<<(unsigned)((p->n_rec + 255) / 256), 256, 0, st>>>(p->n_rec, p->d_crec_seg_off, p->d_cseg_contig, p->d_cseg_start,
                                                                     p->d_cseg_end, p->d_cseg_strand, g->d_contig_len, g->n_contigs,
                                                                     rec, seg);
    MG_LAUNCH_CHECK();
    return MG_OK;
}

extern "C" int mg_plan_predict_cds_device(mg_plan *p, int64_t min_aa, const uint8_t *start64, int flags, mg_cds_pred *rec_out,
                                          mg_cds_seg *seg_out, void *stream) {
    uint64_t start_mask = 0;
    if (const int rc = pred_args(p, flags, start64, &start_mask)) return rc;
    MG_REQUIRE(p->n_rec == 0 || rec_out != nullptr, "rec_out is NULL");
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    p->last_stream = st;
    return pred_launch(p, min_aa, start_mask, flags, rec_out, p->n_cseg > 0 ? seg_out : nullptr, st);
}

extern "C" int mg_plan_predict_cds(mg_plan *p, int64_t min_aa, const uint8_t *start64, int flags, mg_cds_pred *rec_out,
                                   mg_cds_seg *seg_out, void *stream) {
    uint64_t start_mask = 0;
    if (const int rc = pred_args(p, flags, start64, &start_mask)) return rc;
    MG_REQUIRE(p->n_rec == 0 || rec_out != nullptr, "rec_out is NULL");
    if (p->n_rec == 0) return MG_OK;
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    const bool want_seg = seg_out && p->n_cseg > 0;
    if (!p->d_pred || (want_seg && !p->d_pred_seg)) {
        if (const int rc = mg_refuse_growth_in_capture(st, "mg_plan_predict_cds (first call with these outputs)")) return rc;
        auto alloc = [&](void **d, int64_t bytes) -> int {
            MG_CUDA(cudaMallocAsync(d, std::max<int64_t>(bytes, 1), st));
            p->owned.push_back(*d);
            return MG_OK;
        };
        if (!p->d_pred) if (const int rc = alloc((void **)&p->d_pred, p->n_rec * (int64_t)sizeof(mg_cds_pred))) return rc;
        if (want_seg && !p->d_pred_seg) if (const int rc = alloc((void **)&p->d_pred_seg, p->n_cseg * (int64_t)sizeof(mg_cds_seg))) return rc;
    }
    p->last_stream = st;
    if (const int rc = pred_launch(p, min_aa, start_mask, flags, p->d_pred, want_seg ? p->d_pred_seg : nullptr, st)) return rc;
    MG_CUDA(cudaMemcpyAsync(rec_out, p->d_pred, p->n_rec * sizeof(mg_cds_pred), cudaMemcpyDeviceToHost, st));
    if (want_seg) MG_CUDA(cudaMemcpyAsync(seg_out, p->d_pred_seg, p->n_cseg * sizeof(mg_cds_seg), cudaMemcpyDeviceToHost, st));
    return MG_OK;
}
