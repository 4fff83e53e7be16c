// mg_variant.cu -- coding consequences of sorted variant alleles on a prepared plan (mg_plan_variant_count / _emit*).
// Semantics: include/magot_b200.h.
//
// The count queues five launches and reads two results back:
//   k_var_norm   thread per allele: status (contig, bounds, REF against the forward plane, empty / equal alleles), then the
//                suffix-then-prefix trim that gives the forward span [s, t) of REF' and the bytes of A'; the longest REF of an
//                allele with status 0 goes to one atomicMax per warp, which bounds the searches of the join;
//   k_var_join   thread per caller segment e (twice: count, then write): binary searches of the sorted alleles around the
//                segment with its donor site and around its acceptor site, the exact touch test, and ownership (no earlier
//                segment of the record touches the allele, directly or through its junction's sites).  The pairs a segment
//                owns are written in allele order at its offset from mg_scan_i32 (block scan + decoupled look-back);
//   k_var_merge  thread per record: merges its segments' allele-ordered runs into one allele-ordered run.
// The emit is one launch, k_var_emit, thread per row: it walks the row's record once (payload offset of the owning segment,
// the splice sites and the segments the span lies in), and for a substitution gathers every affected codon through the plan's
// pieces (K3's generic gather) and substitutes A' (reverse-complemented on '-').
// The splice-site geometry is a copy of k_check_junctions' rule (mg_check.cu) without the genome read: only whether the junction
// has class 1..4, which does not depend on the bases.  Every genome and payload index is 64-bit.
#include <algorithm>
#include <climits>
#include <cstring>
#include "mg_common.cuh"
#include "mg_gather.cuh"

#define VAR_THREADS 256

static_assert(sizeof(mg_var_effect) == 64, "mg_var_effect layout (include/magot_b200.h)");

struct mg_var_state {
    int64_t n_var = 0, n_rows = 0;
    bool valid = false;                       // a count finished on this plan
    uint64_t generation = 0, prepares = 0;    // genome generation and plan prepare number of that count
    uint64_t start_mask = 0;
    int use_phase = 0;
    // device buffers and their capacities (elements)
    int32_t *contig = nullptr; int64_t *pos = nullptr, *aoff = nullptr; uint8_t *bytes = nullptr;
    int8_t *status = nullptr; int64_t *s = nullptr, *t = nullptr, *alt_lo = nullptr; int32_t *alt_len = nullptr;
    unsigned long long *max_ref = nullptr;
    int32_t *cnt = nullptr; int64_t *seg_off = nullptr, *scan_tmp = nullptr, *cur = nullptr;
    int64_t *pair = nullptr, *row_var = nullptr, *row_seg = nullptr;
    mg_var_effect *out = nullptr;
    int64_t cap_var = 0, cap_bytes = 0, cap_seg = 0, cap_scan = 0, cap_rows = 0, cap_out = 0;
};

struct VarSeg {                                       // one caller segment, clamped as the plan clamps it
    int32_t c;
    bool minus;
    int64_t cl, ch;
};

struct VarArgs {
    const int64_t *crec_seg_off;
    const int32_t *seg_contig;
    const int64_t *seg_start, *seg_end;
    const int8_t *seg_strand;
    const int64_t *contig_len, *contig_base;
    int64_t n_contigs, n_rec, n_seg, n_var;
    const int32_t *contig;
    const int64_t *pos, *aoff;
    const uint8_t *bytes;
    int8_t *status;
    int64_t *s, *t, *alt_lo;
    int32_t *alt_len;
    unsigned long long *max_ref;
};

__device__ __forceinline__ VarSeg var_seg(const VarArgs &a, int64_t e) {
    VarSeg g;
    g.c = __ldg(a.seg_contig + e);                    // contig[start-1:end] with Python slice semantics, as the plan kernels
    g.minus = __ldg(a.seg_strand + e) != 0;
    g.cl = g.ch = 0;
    if (g.c >= 0 && g.c < a.n_contigs) {
        const int64_t L = __ldg(a.contig_len + g.c);
        int64_t i = __ldg(a.seg_start + e) - 1, j = __ldg(a.seg_end + e);
        if (i < 0) { i += L; if (i < 0) i = 0; } else if (i > L) i = L;
        if (j < 0) { j += L; if (j < 0) j = 0; } else if (j > L) j = L;
        g.cl = i;
        g.ch = j > i ? j : i;
    }
    return g;
}

// junction after segment `x` (followed by `y` in the same record) has a class 1..4 in k_check_junctions: both non-empty, same
// contig and strand, intron of at least 4 bases.  Donor site [du, du + 2) shares point dsh with x, acceptor site [au, au + 2)
// shares point ash with y.
__device__ __forceinline__ bool var_sites(const VarSeg &x, const VarSeg &y, int64_t &du, int64_t &dsh, int64_t &au, int64_t &ash) {
    if (!(x.ch > x.cl && y.ch > y.cl && x.c == y.c && x.minus == y.minus)) return false;
    if (!x.minus) {
        if (y.cl - x.ch < 4) return false;
        du = x.ch; dsh = x.ch; au = y.cl - 2; ash = y.cl;
    } else {
        if (x.cl - y.ch < 4) return false;
        du = x.cl - 2; dsh = x.cl; au = y.ch; ash = y.ch;
    }
    return true;
}

__device__ __forceinline__ bool var_touch_seg(int64_t s, int64_t t, const VarSeg &g) {
    return t > s ? (s < g.ch && g.cl < t) : (g.cl < s && s < g.ch);
}

__device__ __forceinline__ bool var_touch_site(int64_t s, int64_t t, int64_t u, int64_t sh) {
    return t > s ? (s < u + 2 && u < t) : (s == u + 1 || s == sh);
}

// does allele (c, [s, t)) touch segment e of a record ending at e1, directly or through junction e's sites
__device__ __forceinline__ bool var_touch_unit(const VarArgs &a, int64_t e, int64_t e1, int32_t c, int64_t s, int64_t t) {
    const VarSeg x = var_seg(a, e);
    if (x.c != c) return false;
    if (var_touch_seg(s, t, x)) return true;
    if (e + 1 >= e1) return false;
    int64_t du, dsh, au, ash;
    if (!var_sites(x, var_seg(a, e + 1), du, dsh, au, ash)) return false;
    return var_touch_site(s, t, du, dsh) || var_touch_site(s, t, au, ash);
}

// first allele index i with (contig[i], pos[i]) >= (c, x)
__device__ __forceinline__ int64_t var_lower(const VarArgs &a, int32_t c, int64_t x) {
    int64_t lo = 0, hi = a.n_var;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int32_t cm = __ldg(a.contig + mid);
        if (cm < c || (cm == c && __ldg(a.pos + mid) < x)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// genome nibble -> upper-case byte: ACGTacgt -> ACGT, N n -> N, then - R Y K M; the exception code 15 gives 0, which no REF
// byte matches
__device__ __forceinline__ uint8_t var_dec(uint32_t nib) {
    const uint64_t lo = 0x5447434154474341ull, hi = 0x004D4B59522D4E4Eull;
    return (uint8_t)(((nib < 8 ? lo : hi) >> (8 * (nib & 7u))) & 0xFFu);
}

__device__ __forceinline__ uint8_t var_upper(uint8_t b) { return (b >= 'a' && b <= 'z') ? (uint8_t)(b - 32) : b; }

__global__ void __launch_bounds__(VAR_THREADS) k_var_norm(const __grid_constant__ VarArgs a, const uint32_t *__restrict__ packed) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    unsigned long long keep = 0;                       // REF length of an allele with status 0, for the warp's max
    if (i < a.n_var) {
        const int32_t c = __ldg(a.contig + i);
        const int64_t p = __ldg(a.pos + i);
        const int64_t r0 = __ldg(a.aoff + 2 * i), r1 = __ldg(a.aoff + 2 * i + 1), a1 = __ldg(a.aoff + 2 * i + 2);
        const int64_t lr = r1 - r0, la = a1 - r1;
        const uint8_t *R = a.bytes + r0, *A = a.bytes + r1;
        int st = 0;
        if (c < 0 || c >= a.n_contigs || p < 0 || p + lr > __ldg(a.contig_len + c)) {
            st = 1;
        } else {
            const int64_t g0 = __ldg(a.contig_base + c) + p;
            uint64_t w = 0;
            for (int64_t k = 0; k < lr; k++) {
                if ((k & 15) == 0) w = mg_ld_nib16(packed, g0 + k);
                const uint32_t nib = (uint32_t)(w >> (4 * (k & 15))) & 15u;
                const uint8_t gb = var_dec(nib);
                if (gb == 0 || gb != var_upper(R[k])) { st = 2; break; }
            }
        }
        int64_t pre = 0, suf = 0;
        if (st == 0) {
            if (lr == 0 || la == 0) {
                st = 3;
            } else {
                const int64_t m = lr < la ? lr : la;
                while (suf < m && var_upper(R[lr - 1 - suf]) == var_upper(A[la - 1 - suf])) suf++;
                while (pre < m - suf && var_upper(R[pre]) == var_upper(A[pre])) pre++;
                if (lr == la && suf == lr) st = 3;      // REF equals ALT ignoring case
            }
        }
        a.status[i] = (int8_t)st;
        if (st == 0) {
            a.s[i] = p + pre;
            a.t[i] = p + lr - suf;
            a.alt_lo[i] = r1 + pre;
            a.alt_len[i] = (int32_t)(la - suf - pre);
            keep = (unsigned long long)lr;
        }
    }
    // one atomic per warp: a single global maximum taken by every allele serialises on one address
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) keep = max(keep, __shfl_xor_sync(0xffffffffu, keep, d));
    if ((threadIdx.x & 31) == 0 && keep) atomicMax(a.max_ref, keep);
}

// visit, in allele order, every allele with status 0 that segment e owns for its record; WRITE: store them from out on
template <bool WRITE>
__global__ void __launch_bounds__(VAR_THREADS) k_var_join(const __grid_constant__ VarArgs a, int32_t *__restrict__ cnt,
                                                          const int64_t *__restrict__ seg_off, int64_t *__restrict__ pair) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= a.n_seg) return;
    const int64_t r = mg_search_le(a.crec_seg_off, 0, a.n_rec, e);
    const int64_t e0 = __ldg(a.crec_seg_off + r), e1 = __ldg(a.crec_seg_off + r + 1);
    const VarSeg x = var_seg(a, e);
    int64_t n = 0;
    if (x.ch > x.cl && a.n_var > 0) {
        const int64_t mr = (int64_t)*a.max_ref;
        // window 1: the segment and its donor site (both strands: within [cl - 2, ch + 2)); window 2: the acceptor site.
        // An allele at pos with REF length lr <= mr spans at most [pos, pos + lr), an insertion sits at pos..pos + lr.
        int64_t w[4];
        w[0] = var_lower(a, x.c, x.cl - 2 - mr - 1);
        w[1] = var_lower(a, x.c, x.ch + 3);
        w[2] = w[3] = w[1];
        int64_t du, dsh, au, ash;
        if (e + 1 < e1 && var_sites(x, var_seg(a, e + 1), du, dsh, au, ash)) {
            w[2] = var_lower(a, x.c, au - mr - 1);
            w[3] = var_lower(a, x.c, au + 3);
        }
        if (w[2] < w[0]) { int64_t t0 = w[0], t1 = w[1]; w[0] = w[2]; w[1] = w[3]; w[2] = t0; w[3] = t1; }
        if (w[2] < w[1]) w[2] = w[1];                   // the two index ranges in order, without overlap
        int64_t out = WRITE ? seg_off[e] : 0;
        for (int k = 0; k < 2; k++) {
            for (int64_t i = w[2 * k]; i < w[2 * k + 1]; i++) {
                if (a.status[i] != 0) continue;
                const int64_t s = a.s[i], t = a.t[i];
                if (!var_touch_unit(a, e, e1, x.c, s, t)) continue;
                bool owned = true;
                for (int64_t q = e0; q < e && owned; q++) owned = !var_touch_unit(a, q, e1, x.c, s, t);
                if (!owned) continue;
                if (WRITE) pair[out++] = i;
                n++;
            }
        }
    }
    if (!WRITE) cnt[e] = (int32_t)n;
}

// each record's rows in allele order: a merge of its segments' runs [seg_off[e], seg_off[e + 1]), cursors in `cur`
__global__ void __launch_bounds__(VAR_THREADS) k_var_merge(int64_t n_rec, const int64_t *__restrict__ crec_seg_off,
                                                           const int64_t *__restrict__ seg_off, const int64_t *__restrict__ pair,
                                                           int64_t *__restrict__ cur, int64_t *__restrict__ row_var,
                                                           int64_t *__restrict__ row_seg) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const int64_t e0 = crec_seg_off[r], e1 = crec_seg_off[r + 1];
    if (e1 <= e0) return;
    const int64_t k0 = seg_off[e0], k1 = seg_off[e1];
    int nonempty = 0;
    for (int64_t e = e0; e < e1; e++) {
        cur[e] = seg_off[e];
        nonempty += seg_off[e + 1] > seg_off[e];
    }
    if (nonempty <= 1) {                               // one run: already in order
        for (int64_t e = e0; e < e1; e++)
            for (int64_t k = seg_off[e]; k < seg_off[e + 1]; k++) { row_var[k] = pair[k]; row_seg[k] = e; }
        return;
    }
    for (int64_t k = k0; k < k1; k++) {
        int64_t best = -1, bv = LLONG_MAX;
        for (int64_t e = e0; e < e1; e++) {
            const int64_t c = cur[e];
            if (c < seg_off[e + 1] && pair[c] < bv) { bv = pair[c]; best = e; }
        }
        row_var[k] = bv;
        row_seg[k] = best;
        cur[best]++;
    }
}

struct VarEmitArgs {
    VarArgs v;
    const uint32_t *packed;
    const int64_t *piece_off, *piece_src, *rec_seg_off;
    const int8_t *rec_phase;
    const uint8_t *aa4096;                             // the plan's code: nibble triplet (first base lowest) -> residue
    uint64_t stop_mask, start_mask;
    int use_phase;
    int64_t n_rows;
    const int64_t *row_var, *row_seg;
    mg_var_effect *out;
};

// 2-bit base of an ALT byte, 8 = outside A/C/G/T
__device__ __forceinline__ uint32_t var_alt_code(uint8_t b) {
    switch (b) {
    case 'A': case 'a': return 0; case 'C': case 'c': return 1; case 'G': case 'g': return 2; case 'T': case 't': return 3;
    default: return 8;
    }
}

__global__ void __launch_bounds__(VAR_THREADS) k_var_emit(const __grid_constant__ VarEmitArgs a) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= a.n_rows) return;
    const VarArgs &v = a.v;
    const int64_t i = a.row_var[k], eo = a.row_seg[k];
    const int64_t r = mg_search_le(v.crec_seg_off, 0, v.n_rec, eo);
    const int64_t e0 = __ldg(v.crec_seg_off + r), e1 = __ldg(v.crec_seg_off + r + 1);
    const int32_t c = __ldg(v.contig + i);
    const int64_t s = v.s[i], t = v.t[i], alt_lo = v.alt_lo[i];
    const int64_t la = v.alt_len[i], lr = t - s;
    // one walk over the record: sites touched, whether [s, t) lies in one segment, the owning segment's payload offset
    bool acc = false, don = false, inside = false;
    int64_t o = 0, oo = 0, len = 0;
    VarSeg xo = var_seg(v, eo);
    VarSeg x = var_seg(v, e0);
    for (int64_t e = e0; e < e1; e++) {
        if (e == eo) oo = o;
        if (x.c == c && (lr > 0 ? (x.cl <= s && t <= x.ch) : (x.cl < s && s < x.ch))) inside = true;
        VarSeg y;
        if (e + 1 < e1) {
            y = var_seg(v, e + 1);
            int64_t du, dsh, au, ash;
            if (x.c == c && var_sites(x, y, du, dsh, au, ash)) {
                don |= var_touch_site(s, t, du, dsh);
                acc |= var_touch_site(s, t, au, ash);
            }
        }
        o += x.ch - x.cl;
        x = y;
    }
    len = o;
    int skip = a.use_phase && a.rec_phase ? a.rec_phase[r] : 0;
    if (skip < 0 || skip > 2) skip = 0;
    const int64_t L = len - skip, ncod = L > 0 ? L / 3 : 0;
    const int64_t cod_lo = skip, cod_hi = skip + 3 * ncod;
    // payload range of the span's part in the owning segment
    int64_t nlo = -1, nhi = -1;
    if (lr > 0) {
        const int64_t x0 = max(s, xo.cl), x1 = min(t, xo.ch);
        if (x0 < x1) {
            if (xo.minus) { nlo = oo + xo.ch - x1; nhi = oo + xo.ch - x0; }
            else { nlo = oo + x0 - xo.cl; nhi = oo + x1 - xo.cl; }
        }
    } else if (xo.cl < s && s < xo.ch) {
        nlo = nhi = xo.minus ? oo + xo.ch - s : oo + s - xo.cl;
    }
    const bool sub = lr == la;
    mg_var_effect out;
    out.var = i;
    out.rec = r;
    out.seg = eo;
    out.nuc_lo = nlo;
    out.nuc_hi = nhi;
    out.codon = -1;
    out.n_aff = 0;
    out.ref_codon = out.alt_codon = 0xFF;
    uint64_t raa = 0, aaa = 0;                          // ref_aa / alt_aa, residue m in byte m
    int64_t ia = 0, ib = -1;                            // affected codons of a substitution: [ia, ib]
    if (nlo >= 0) {
        if (sub) {
            const int64_t x0 = max(nlo, cod_lo), x1 = min(nhi, cod_hi);
            if (x0 < x1) { ia = (x0 - skip) / 3; ib = (x1 - 1 - skip) / 3; out.codon = (int32_t)ia; }
        } else if (nlo >= cod_lo && nlo < cod_hi) {
            out.codon = (int32_t)((nlo - skip) / 3);
        }
    }
    int cls;
    if (acc) cls = MG_VEF_SPLICE_ACCEPTOR;
    else if (don) cls = MG_VEF_SPLICE_DONOR;
    else if (!inside) cls = MG_VEF_BOUNDARY;
    else if (!sub) {
        const int64_t d = la - lr;
        cls = d % 3 != 0 ? MG_VEF_FRAMESHIFT : (d > 0 ? MG_VEF_INFRAME_INSERTION : MG_VEF_INFRAME_DELETION);
    } else if (ib < ia) {
        cls = MG_VEF_NONCODING_PAYLOAD;
    } else {
        const int64_t f0 = __ldg(a.rec_seg_off + r) + 2 * r, f1 = __ldg(a.rec_seg_off + r + 1) + 2 * (r + 1);
        const int64_t ns = __ldg(a.piece_off + f0 + 1);
        bool start_lost = false, stop_gained = false, stop_lost = false, ambig = false, missense = false;
        for (int64_t ci = ia; ci <= ib; ci++) {
            const int64_t P = skip + 3 * ci;
            const int64_t j = mg_search_le(a.piece_off, f0 + 1, f1 - 1, ns + P);
            uint64_t g3[3];
            mg_gather_nib(a.packed, a.piece_off, a.piece_src, j, ns + P, 3, g3);
            uint32_t rb[3], ab[3];
#pragma unroll
            for (int b = 0; b < 3; b++) {
                const uint32_t nib = (uint32_t)(g3[0] >> (4 * b)) & 15u;
                rb[b] = nib < 8 ? (nib & 3u) : 8u;
                const int64_t q = P + b;
                if (q >= nlo && q < nhi) {
                    const int64_t kk = q - nlo;
                    if (xo.minus) { const uint32_t cb = var_alt_code(v.bytes[alt_lo + la - 1 - kk]); ab[b] = cb < 4 ? (cb ^ 3u) : 8u; }
                    else ab[b] = var_alt_code(v.bytes[alt_lo + kk]);
                } else {
                    ab[b] = rb[b];
                }
            }
            const bool ra = (rb[0] | rb[1] | rb[2]) & 8u, aa = (ab[0] | ab[1] | ab[2]) & 8u;
            const uint32_t ri = ra ? 0xFFu : (rb[0] << 4 | rb[1] << 2 | rb[2]);
            const uint32_t ai = aa ? 0xFFu : (ab[0] << 4 | ab[1] << 2 | ab[2]);
            const uint8_t rres = ra ? (uint8_t)'X' : __ldg(a.aa4096 + (rb[0] | rb[1] << 4 | rb[2] << 8));
            const uint8_t ares = aa ? (uint8_t)'X' : __ldg(a.aa4096 + (ab[0] | ab[1] << 4 | ab[2] << 8));
            const bool rstop = !ra && ((a.stop_mask >> ri) & 1), astop = !aa && ((a.stop_mask >> ai) & 1);
            if (ci == 0 && !ra && ((a.start_mask >> ri) & 1) && !(!aa && ((a.start_mask >> ai) & 1))) start_lost = true;
            if (!ra && !rstop && astop) stop_gained = true;
            if (ci == ncod - 1 && rstop && !astop) stop_lost = true;
            if (ra || aa) ambig = true;
            else if (rres != ares) missense = true;
            const int64_t m = ci - ia;
            if (m == 0) { out.ref_codon = (uint8_t)ri; out.alt_codon = (uint8_t)ai; }
            if (m < 8) { raa |= (uint64_t)rres << (8 * m); aaa |= (uint64_t)ares << (8 * m); }
        }
        out.n_aff = (int8_t)min(ib - ia + 1, (int64_t)127);
        cls = start_lost ? MG_VEF_START_LOST : stop_gained ? MG_VEF_STOP_GAINED : stop_lost ? MG_VEF_STOP_LOST
              : ambig ? MG_VEF_AMBIGUOUS : missense ? MG_VEF_MISSENSE : MG_VEF_SYNONYMOUS;
    }
    out.cls = (int8_t)cls;
    memcpy(out.ref_aa, &raa, 8);
    memcpy(out.alt_aa, &aaa, 8);
    a.out[k] = out;
}

// ---- host API -----------------------------------------------------------------------------------------------

static int var_alloc(void **d, int64_t bytes, cudaStream_t st) {
    if (*d) MG_CUDA(cudaFreeAsync(*d, st));
    *d = nullptr;
    MG_CUDA(cudaMallocAsync(d, std::max<int64_t>(bytes, 1), st));
    return MG_OK;
}

void mg_var_free(mg_plan *p) {
    mg_var_state *v = p->var;
    if (!v) return;
    cudaStream_t st = p->last_stream;
    void *bufs[] = {v->contig, v->pos, v->aoff, v->bytes, v->status, v->s, v->t, v->alt_lo, v->alt_len, v->max_ref, v->cnt,
                    v->seg_off, v->scan_tmp, v->cur, v->pair, v->row_var, v->row_seg, v->out};
    for (void *b : bufs) if (b) cudaFreeAsync(b, st);
    delete v;
    p->var = nullptr;
}

static VarArgs var_args(mg_plan *p) {
    mg_genome *g = p->g;
    mg_var_state *v = p->var;
    VarArgs a;
    a.crec_seg_off = p->d_crec_seg_off; a.seg_contig = p->d_cseg_contig; a.seg_start = p->d_cseg_start; a.seg_end = p->d_cseg_end;
    a.seg_strand = p->d_cseg_strand; a.contig_len = g->d_contig_len; a.contig_base = g->d_contig_base; a.n_contigs = g->n_contigs;
    a.n_rec = p->n_rec; a.n_seg = p->n_cseg; a.n_var = v->n_var;
    a.contig = v->contig; a.pos = v->pos; a.aoff = v->aoff; a.bytes = v->bytes; a.status = v->status;
    a.s = v->s; a.t = v->t; a.alt_lo = v->alt_lo; a.alt_len = v->alt_len; a.max_ref = v->max_ref;
    return a;
}

static unsigned var_blocks(int64_t n) { return (unsigned)((n + VAR_THREADS - 1) / VAR_THREADS); }

extern "C" int mg_plan_variant_count(mg_plan *p, int64_t n_var, const int32_t *contig, const int64_t *pos, const int64_t *allele_off,
                                     const uint8_t *bytes, int64_t n_bytes, int flags, const uint8_t *start64, int8_t *status_host,
                                     int64_t *n_rows, void *stream) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    MG_REQUIRE((flags & ~MG_PROT_USE_PHASE) == 0, "flags: only MG_PROT_USE_PHASE is accepted");
    MG_REQUIRE(n_var >= 0 && n_bytes >= 0, "n_var and n_bytes must be >= 0");
    MG_REQUIRE(n_rows != nullptr, "n_rows is NULL");
    MG_REQUIRE(n_var == 0 || (contig && pos && allele_off && status_host), "an allele array is NULL");
    MG_REQUIRE(n_bytes == 0 || bytes != nullptr, "bytes is NULL");
    uint64_t start_mask = 0;
    if (const int rc = mg_start_mask(p, start64, &start_mask)) return rc;
    if (const int rc = mg_plan_check_prepared(p)) return rc;
    if (n_var > 0) {
        MG_REQUIRE(allele_off[0] >= 0 && allele_off[2 * n_var] <= n_bytes, "allele_off runs outside bytes");
        for (int64_t k = 0; k < 2 * n_var; k++) MG_REQUIRE(allele_off[k] <= allele_off[k + 1], "allele_off is not non-decreasing");
        for (int64_t i = 1; i < n_var; i++)
            MG_REQUIRE(contig[i - 1] < contig[i] || (contig[i - 1] == contig[i] && pos[i - 1] <= pos[i]),
                       "alleles are not sorted by (contig, pos)");
    }
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (const int rc = mg_refuse_growth_in_capture(st, "mg_plan_variant_count (returns a row count to the host)")) return rc;
    if (!p->var) p->var = new mg_var_state();
    mg_var_state *v = p->var;
    v->valid = false;
    p->last_stream = st;
    *n_rows = 0;
    v->n_var = n_var;
    int rc;
    if (n_var > v->cap_var || !v->contig) {
        const int64_t n = std::max<int64_t>(n_var, 1);
        if ((rc = var_alloc((void **)&v->contig, n * 4, st)) || (rc = var_alloc((void **)&v->pos, n * 8, st)) ||
            (rc = var_alloc((void **)&v->aoff, (2 * n + 1) * 8, st)) || (rc = var_alloc((void **)&v->status, n, st)) ||
            (rc = var_alloc((void **)&v->s, n * 8, st)) || (rc = var_alloc((void **)&v->t, n * 8, st)) ||
            (rc = var_alloc((void **)&v->alt_lo, n * 8, st)) || (rc = var_alloc((void **)&v->alt_len, n * 4, st)))
            return rc;
        v->cap_var = n;
    }
    if (n_bytes > v->cap_bytes || !v->bytes) {
        if ((rc = var_alloc((void **)&v->bytes, n_bytes, st))) return rc;
        v->cap_bytes = std::max<int64_t>(n_bytes, 1);
    }
    const int64_t n_seg = p->n_cseg;
    const int64_t scan_need = mg_scan_tmp_elems(n_seg);
    if (n_seg > v->cap_seg || !v->cnt) {
        const int64_t n = std::max<int64_t>(n_seg, 1);
        if ((rc = var_alloc((void **)&v->cnt, n * 4, st)) || (rc = var_alloc((void **)&v->seg_off, (n + 1) * 8, st)) ||
            (rc = var_alloc((void **)&v->cur, n * 8, st)))
            return rc;
        v->cap_seg = n;
    }
    if (scan_need > v->cap_scan || !v->scan_tmp) {
        if ((rc = var_alloc((void **)&v->scan_tmp, scan_need * 8, st))) return rc;
        v->cap_scan = scan_need;
    }
    if (!v->max_ref && (rc = var_alloc((void **)&v->max_ref, 8, st))) return rc;
    if (n_var > 0) {
        MG_CUDA(cudaMemcpyAsync(v->contig, contig, n_var * 4, cudaMemcpyHostToDevice, st));
        MG_CUDA(cudaMemcpyAsync(v->pos, pos, n_var * 8, cudaMemcpyHostToDevice, st));
        MG_CUDA(cudaMemcpyAsync(v->aoff, allele_off, (2 * n_var + 1) * 8, cudaMemcpyHostToDevice, st));
        if (n_bytes > 0) MG_CUDA(cudaMemcpyAsync(v->bytes, bytes, n_bytes, cudaMemcpyHostToDevice, st));
    }
    MG_CUDA(cudaMemsetAsync(v->max_ref, 0, 8, st));
    const VarArgs a = var_args(p);
    if (n_var > 0) {
        k_var_norm<<<var_blocks(n_var), VAR_THREADS, 0, st>>>(a, p->g->d_packed);
        MG_LAUNCH_CHECK();
    }
    int64_t total = 0;
    if (n_seg > 0) {
        k_var_join<false><<<var_blocks(n_seg), VAR_THREADS, 0, st>>>(a, v->cnt, nullptr, nullptr);
        MG_LAUNCH_CHECK();
        if ((rc = mg_scan_i32(v->cnt, v->seg_off, n_seg, v->scan_tmp, v->cap_scan, st))) return rc;
        MG_CUDA(cudaMemcpyAsync(&total, v->seg_off + n_seg, 8, cudaMemcpyDeviceToHost, st));
    }
    if (n_var > 0) MG_CUDA(cudaMemcpyAsync(status_host, v->status, n_var, cudaMemcpyDeviceToHost, st));
    MG_CUDA(cudaStreamSynchronize(st));
    if (total > 0) {
        if (total > v->cap_rows || !v->pair) {
            if ((rc = var_alloc((void **)&v->pair, total * 8, st)) || (rc = var_alloc((void **)&v->row_var, total * 8, st)) ||
                (rc = var_alloc((void **)&v->row_seg, total * 8, st)))
                return rc;
            v->cap_rows = total;
        }
        k_var_join<true><<<var_blocks(n_seg), VAR_THREADS, 0, st>>>(a, v->cnt, v->seg_off, v->pair);
        MG_LAUNCH_CHECK();
        k_var_merge<<<var_blocks(p->n_rec), VAR_THREADS, 0, st>>>(p->n_rec, p->d_crec_seg_off, v->seg_off, v->pair, v->cur,
                                                                   v->row_var, v->row_seg);
        MG_LAUNCH_CHECK();
    }
    v->n_rows = total;
    v->start_mask = start_mask;
    v->use_phase = (flags & MG_PROT_USE_PHASE) != 0;
    v->generation = p->g->generation;
    v->prepares = p->prepares;
    v->valid = true;
    *n_rows = total;
    return MG_OK;
}

static int var_emit_check(mg_plan *p) {
    MG_REQUIRE(p != nullptr, "plan handle is NULL");
    mg_var_state *v = p->var;
    if (!v || !v->valid) { mg_set_error("mg_plan_variant_count has not been called on this plan"); return MG_ESTATE; }
    if (v->prepares != p->prepares || v->generation != p->g->generation) {
        mg_set_error("the plan was prepared again or its genome changed since mg_plan_variant_count: count again");
        return MG_ESTATE;
    }
    return mg_plan_check_prepared(p);
}

static int var_emit_launch(mg_plan *p, mg_var_effect *out, cudaStream_t st) {
    mg_var_state *v = p->var;
    if (v->n_rows == 0) return MG_OK;
    mg_genome *g = p->g;
    VarEmitArgs a;
    a.v = var_args(p);
    a.packed = g->d_packed; a.piece_off = p->d_piece_off; a.piece_src = p->d_piece_src; a.rec_seg_off = p->d_rec_seg_off;
    a.rec_phase = p->d_rec_phase;
    a.aa4096 = p->own_code ? p->d_aa8192 : g->d_aa4096;
    a.stop_mask = p->stop_mask; a.start_mask = v->start_mask; a.use_phase = v->use_phase;
    a.n_rows = v->n_rows; a.row_var = v->row_var; a.row_seg = v->row_seg; a.out = out;
    k_var_emit<<<var_blocks(v->n_rows), VAR_THREADS, 0, st>>>(a);
    MG_LAUNCH_CHECK();
    return MG_OK;
}

extern "C" int mg_plan_variant_emit_device(mg_plan *p, mg_var_effect *rows_dev, void *stream) {
    if (const int rc = var_emit_check(p)) return rc;
    MG_REQUIRE(p->var->n_rows == 0 || rows_dev != nullptr, "rows_dev is NULL");
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    p->last_stream = st;
    return var_emit_launch(p, rows_dev, st);
}

extern "C" int mg_plan_variant_emit(mg_plan *p, mg_var_effect *rows_host, void *stream) {
    if (const int rc = var_emit_check(p)) return rc;
    mg_var_state *v = p->var;
    MG_REQUIRE(v->n_rows == 0 || rows_host != nullptr, "rows_host is NULL");
    if (v->n_rows == 0) return MG_OK;
    MG_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    p->last_stream = st;
    if (v->n_rows > v->cap_out || !v->out) {
        if (const int rc = var_alloc((void **)&v->out, v->n_rows * (int64_t)sizeof(mg_var_effect), st)) return rc;
        v->cap_out = v->n_rows;
    }
    if (const int rc = var_emit_launch(p, v->out, st)) return rc;
    MG_CUDA(cudaMemcpyAsync(rows_host, v->out, v->n_rows * sizeof(mg_var_effect), cudaMemcpyDeviceToHost, st));
    return MG_OK;
}
