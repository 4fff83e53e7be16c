// mg_mask.cu -- K5: interval SCATTER on the packed genome (soft / hard masking of annotated intervals).
// Replaces the per-interval list surgery of mask_from_gff (genome_tools.py:394-428):
//     genome_dict[seqid][start-1:stop] = lower(...)      mask_type "soft"
//     genome_dict[seqid][start-1:stop] = 'N' * n         mask_type "hard"
// and its optional upper-casing of the whole genome first (overwrite_softmask, :403-404).
//
// In code space both masks are bit operations on the 4-bit codes (mg_common.cuh), so overlapping or
// duplicate intervals need no ordering: soft = OR (ACGT 0-3 -> acgt: |4, N 8 -> n: |1, RYKM 11-14 ->
// exception code 15: |15, everything else unchanged), hard = AND 0 then OR 8 ('N').  One warp walks
// one interval, 8 bases per lane and step, with atomicOr / atomicAnd on the words, so two intervals
// that share a word cannot lose each other's update.  Lower-cased R/Y/K/M leave the packed alphabet:
// they are listed first (read-only pass, repeatable if the list has to grow) and join the exception
// side list.  Only the forward plane is touched; the reverse-complement plane is rebuilt from it
// afterwards by one streaming pass (1 B/base of HBM traffic), which also keeps its "anything outside
// acgtn- -> n" rule (genome.py:791-792) exact.
#include <algorithm>
#include "mg_common.cuh"

#define NIB1 0x11111111u

// nibble-granular mask of the bases [lo, hi) (global indices) inside the 8-base word that starts at base w0
__device__ __forceinline__ uint32_t word_range_mask(int64_t w0, int64_t lo, int64_t hi) {
    const int a = (int)max((int64_t)0, lo - w0), b = (int)min((int64_t)8, hi - w0);
    if (b <= a) return 0u;
    const uint32_t upto_b = b >= 8 ? 0xFFFFFFFFu : ((1u << (4 * b)) - 1u);
    return upto_b & ~((1u << (4 * a)) - 1u);            // a <= 7 here
}

// flags (bit 0 of each nibble) of the codes 11..14 = R Y K M
__device__ __forceinline__ uint32_t iupac_flags(uint32_t x) {
    const uint32_t b0 = x & NIB1, b1 = (x >> 1) & NIB1, b2 = (x >> 2) & NIB1, b3 = (x >> 3) & NIB1;
    const uint32_t ge11 = b3 & (b2 | (b1 & b0));        // 11, 12..15
    const uint32_t is15 = b3 & b2 & b1 & b0;
    return ge11 & ~is15;
}

// pass 1 of a soft mask: list the R/Y/K/M bases inside the intervals (they become exceptions 'r' 'y' 'k' 'm')
__global__ void __launch_bounds__(256) k_mask_list_iupac(const uint32_t *__restrict__ packed, int64_t n_iv, const int64_t *__restrict__ lo,
                                                         const int64_t *__restrict__ hi, int64_t *__restrict__ out_pos,
                                                         uint8_t *__restrict__ out_byte, int64_t cap, unsigned long long *count) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5, n_warp = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp; i < n_iv; i += n_warp) {
        const int64_t a = lo[i], b = hi[i];
        for (int64_t w0 = (a & ~7ll) + 8ll * lane; w0 < b; w0 += 256) {
            const uint32_t x = __ldg(packed + (w0 >> 3));
            uint32_t f = iupac_flags(x) & word_range_mask(w0, a, b);
            while (f) {
                const int k = (__ffs(f) - 1) >> 2;
                f &= f - 1;
                const unsigned long long slot = atomicAdd(count, 1ull);
                if ((int64_t)slot < cap) {
                    out_pos[slot] = w0 + k;
                    out_byte[slot] = (uint8_t)("rykm"[((x >> (4 * k)) & 15u) - 11u]);
                }
            }
        }
    }
}

// pass 2: the mask itself.  mode 0 = soft, 1 = hard
__global__ void __launch_bounds__(256) k_mask_apply(uint32_t *__restrict__ packed, int64_t n_iv, const int64_t *__restrict__ lo,
                                                    const int64_t *__restrict__ hi, int mode) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5, n_warp = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp; i < n_iv; i += n_warp) {
        const int64_t a = lo[i], b = hi[i];
        for (int64_t w0 = (a & ~7ll) + 8ll * lane; w0 < b; w0 += 256) {
            uint32_t *p = packed + (w0 >> 3);
            const uint32_t m = word_range_mask(w0, a, b);
            if (mode == 1) {
                atomicAnd(p, ~m);
                atomicOr(p, 0x88888888u & m);
            } else {
                const uint32_t x = *p;
                const uint32_t b0 = x & NIB1, b1 = (x >> 1) & NIB1, b2 = (x >> 2) & NIB1, b3 = (x >> 3) & NIB1;
                const uint32_t acgt = NIB1 & ~b3 & ~b2;                          // 0..3  -> set bit 2
                const uint32_t isN = b3 & ~b2 & ~b1 & ~b0;                        // 8     -> set bit 0
                const uint32_t orv = ((acgt << 2) | isN | (iupac_flags(x) * 15u)) & m;
                if (orv) atomicOr(p, orv);
            }
        }
    }
}

// upper-case the whole forward plane: acgt 4..7 -> ACGT (clear bit 2), n 9 -> N (clear bit 0)
__global__ void __launch_bounds__(256) k_mask_upper(uint32_t *__restrict__ packed, int64_t w_lo, int64_t w_hi) {
    for (int64_t w = w_lo + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w < w_hi; w += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t x = packed[w];
        const uint32_t b0 = x & NIB1, b1 = (x >> 1) & NIB1, b2 = (x >> 2) & NIB1, b3 = (x >> 3) & NIB1;
        const uint32_t lower = ~b3 & b2 & NIB1, is9 = b3 & ~b2 & ~b1 & b0;
        const uint32_t y = x & ~(lower << 2) & ~is9;
        if (y != x) packed[w] = y;
    }
}

// reverse-complement plane from the forward plane: word W of the second plane mirrors word 2T/8 - 1 - W
__global__ void __launch_bounds__(256) k_mask_rebuild_rc(uint32_t *__restrict__ packed, int64_t words_per_plane) {
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < words_per_plane; j += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t f = packed[words_per_plane - 1 - j];
        packed[words_per_plane + j] = mg_comp_nib32(mg_rev_nib32(f));
    }
}

extern "C" int mg_genome_mask(mg_genome *g, int64_t n_iv, const int32_t *contig, const int64_t *lo, const int64_t *hi, int hard,
                              int upper_first, void *stream) {
    MG_REQUIRE(g != nullptr, "genome handle is NULL");
    MG_REQUIRE(g->finalized, "mg_genome_finalize has not been called");
    MG_REQUIRE(n_iv >= 0 && (n_iv == 0 || (contig && lo && hi)), "bad interval table");
    MG_CUDA(cudaSetDevice(g->device));
    cudaStream_t st = (cudaStream_t)stream;
    g->stops_valid = g->stops_alt_valid = false;                          // the stop-codon index of the ORF scan is rebuilt on its next use
    // host: intervals in global base indices
    std::vector<int64_t> glo(n_iv), ghi(n_iv);
    for (int64_t i = 0; i < n_iv; i++) {
        MG_REQUIRE(contig[i] >= 0 && contig[i] < g->n_contigs, "interval on an unknown contig");
        MG_REQUIRE(lo[i] >= 0 && lo[i] <= hi[i] && hi[i] <= g->h_contig_len[contig[i]], "interval outside its contig (clamp it like a Python slice first)");
        glo[i] = g->h_contig_base[contig[i]] + lo[i];
        ghi[i] = g->h_contig_base[contig[i]] + hi[i];
    }
    g->generation++;                                                      // counts and plans from before this call are stale
    const int64_t T = g->total_bases, words = T / 8;
    int64_t *d_lo = nullptr, *d_hi = nullptr;
    if (n_iv) {
        MG_CUDA(cudaMallocAsync((void **)&d_lo, 2 * n_iv * sizeof(int64_t), st));
        d_hi = d_lo + n_iv;
        MG_CUDA(cudaMemcpyAsync(d_lo, glo.data(), n_iv * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        MG_CUDA(cudaMemcpyAsync(d_hi, ghi.data(), n_iv * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    }
    const int grid = 148 * 8;
    if (upper_first) {
        k_mask_upper<<<grid, 256, 0, st>>>(g->d_packed, MG_FRONT_PAD / 8, words);
        MG_LAUNCH_CHECK();
        for (auto &c : g->h_exc_byte) if (c >= 'a' && c <= 'z') c = (uint8_t)(c - 32);       // str.upper(), C locale
    }
    // exceptions that already exist: bytes inside a soft interval are lower-cased, inside a hard interval they vanish
    if (n_iv && !g->h_exc_pos.empty()) {
        std::vector<std::pair<int64_t, int64_t>> iv(n_iv);
        for (int64_t i = 0; i < n_iv; i++) iv[i] = {glo[i], ghi[i]};
        std::sort(iv.begin(), iv.end());
        std::vector<std::pair<int64_t, int64_t>> merged;
        for (auto &v : iv) {
            if (v.second <= v.first) continue;
            if (!merged.empty() && v.first <= merged.back().second) merged.back().second = std::max(merged.back().second, v.second);
            else merged.push_back(v);
        }
        size_t keep = 0;
        for (size_t k = 0; k < g->h_exc_pos.size(); k++) {
            const int64_t pos = g->h_exc_pos[k];
            auto it = std::upper_bound(merged.begin(), merged.end(), std::make_pair(pos, INT64_MAX));
            const bool inside = it != merged.begin() && pos < (it - 1)->second;
            uint8_t c = g->h_exc_byte[k];
            if (inside && hard) continue;
            if (inside && c >= 'A' && c <= 'Z') c = (uint8_t)(c + 32);                          // str.lower()
            g->h_exc_pos[keep] = pos;
            g->h_exc_byte[keep++] = c;
        }
        g->h_exc_pos.resize(keep);
        g->h_exc_byte.resize(keep);
    }
    if (n_iv) {
        if (!hard) {                                   // R/Y/K/M inside the intervals leave the alphabet
            int64_t cap = 1 << 16;
            for (;;) {
                int64_t *d_pos = nullptr;
                uint8_t *d_byte = nullptr;
                MG_CUDA(cudaMallocAsync((void **)&d_pos, cap * sizeof(int64_t), st));
                MG_CUDA(cudaMallocAsync((void **)&d_byte, cap, st));
                MG_CUDA(cudaMemsetAsync(g->d_exc_count, 0, sizeof(unsigned long long), st));
                k_mask_list_iupac<<<grid, 256, 0, st>>>(g->d_packed, n_iv, d_lo, d_hi, d_pos, d_byte, cap, g->d_exc_count);
                MG_LAUNCH_CHECK();
                unsigned long long cnt = 0;
                MG_CUDA(cudaMemcpyAsync(&cnt, g->d_exc_count, sizeof(cnt), cudaMemcpyDeviceToHost, st));
                MG_CUDA(cudaStreamSynchronize(st));
                if ((int64_t)cnt <= cap && cnt) {
                    const size_t old = g->h_exc_pos.size();
                    g->h_exc_pos.resize(old + cnt);
                    g->h_exc_byte.resize(old + cnt);
                    MG_CUDA(cudaMemcpy(g->h_exc_pos.data() + old, d_pos, cnt * sizeof(int64_t), cudaMemcpyDeviceToHost));
                    MG_CUDA(cudaMemcpy(g->h_exc_byte.data() + old, d_byte, cnt, cudaMemcpyDeviceToHost));
                }
                MG_CUDA(cudaFreeAsync(d_pos, st));
                MG_CUDA(cudaFreeAsync(d_byte, st));
                if ((int64_t)cnt <= cap) break;
                cap = (int64_t)cnt + 1024;             // the pass only reads: run it again with room for everything
            }
        }
        k_mask_apply<<<grid, 256, 0, st>>>(g->d_packed, n_iv, d_lo, d_hi, hard ? 1 : 0);
        MG_LAUNCH_CHECK();
        MG_CUDA(cudaFreeAsync(d_lo, st));
    }
    k_mask_rebuild_rc<<<grid, 256, 0, st>>>(g->d_packed, words);
    MG_LAUNCH_CHECK();
    MG_CUDA(cudaStreamSynchronize(st));
    // sorted, de-duplicated exception list back to the device (overlapping intervals list a base twice: same byte)
    return mg_genome_finalize(g, nullptr);
}
