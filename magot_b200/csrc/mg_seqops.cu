// mg_seqops.cu -- Sequence.reverse_compliment (genome.py:784-793) and Sequence.translate
// (genome.py:795-822, all frames / strands / trimX incl. the `(pos + frame) % 3 == 2` quirk) on
// arbitrary ASCII strings handed over by the host; backs the `Sequence` class and cds2pep
// (genome_tools.py:664-675).  Flat passes over output bytes, 16 per thread, like K2/K3.
#include <algorithm>
#include "mg_common.cuh"

// complement of one ASCII byte (genome.py:787, :791-792)
__device__ __forceinline__ uint32_t comp_ascii(uint32_t c) {
    switch (c) {
    case 'a': return 't'; case 't': return 'a'; case 'g': return 'c'; case 'c': return 'g';
    case 'A': return 'T'; case 'T': return 'A'; case 'G': return 'C'; case 'C': return 'G';
    case 'n': return 'n'; case 'N': return 'N'; case '-': return '-';
    default: return 'n';
    }
}

__global__ void __launch_bounds__(256) k_revcomp_ascii(const uint8_t *__restrict__ in, int64_t n, uint8_t *__restrict__ out) {
    const int64_t nchunk = (n + 15) >> 4;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nchunk; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o = i << 4;
        uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
        for (int k = 0; k < 16; k++) {
            if (o + k < n) w[k >> 2] |= comp_ascii(__ldg(in + (n - 1 - o - k))) << ((k & 3) * 8);
        }
        mg_st16(out + o, w[0], w[1], w[2], w[3]);
    }
}

// 2-bit class of an ASCII base after .upper() (genome.py:812): A=0 C=1 G=2 T=3, anything else 8
__device__ __forceinline__ uint32_t base_code(uint32_t c) {
    switch (c) {
    case 'A': case 'a': return 0; case 'C': case 'c': return 1;
    case 'G': case 'g': return 2; case 'T': case 't': return 3;
    default: return 8;
    }
}

// oriented base q of a sequence of length L starting at `s` (minus: complement of base L-1-q)
__device__ __forceinline__ uint32_t oriented_code(const uint8_t *__restrict__ s, int64_t L, int64_t q, int minus) {
    if (!minus) return base_code(__ldg(s + q));
    const uint32_t c = base_code(__ldg(s + (L - 1 - q)));
    return c < 8 ? (c ^ 3u) : c;
}

// translate geometry for (frame, L): `lead` = 1 when the reference emits an artificial 'X' for the partial
// first triplet (frames 1 and 2), cs = offset of the first full codon, nfull = number of full codons.
__device__ __forceinline__ void tr_geometry(int frame, int64_t L, int &lead, int64_t &cs, int64_t &nfull) {
    if (frame == 0) { lead = 0; cs = 0; nfull = L / 3; }
    else if (frame == 1) { lead = 1; cs = 2; nfull = (L + 1) / 3 - 1; }   // emits at pos 1,4,7,..
    else { lead = 1; cs = 4; nfull = (L - 1) / 3 - 1; }                     // emits at pos 3,6,9,..
}

// pass 1: output length of every sequence (-1 = the reference returns None, genome.py:810)
__global__ void __launch_bounds__(256) k_tr_len(const uint8_t *__restrict__ in, const int64_t *__restrict__ off, int64_t n_seq,
                                                int frame, int minus, int trimX, const uint8_t *__restrict__ aa4096,
                                                int32_t *__restrict__ len32, int64_t *__restrict__ out_len, int8_t *__restrict__ drop) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_seq) return;
    const int64_t L = off[i + 1] - off[i];
    if (!(L > 2 + frame)) { len32[i] = 0; out_len[i] = -1; drop[i] = 0; return; }
    int lead; int64_t cs, nfull;
    tr_geometry(frame, L, lead, cs, nfull);
    int64_t m = lead + nfull;
    int d = 0;
    if (trimX) {
        if (lead) d = 1;                                  // the artificial X is always trimmed
        else {
            const uint8_t *s = in + off[i];
            const uint32_t idx = oriented_code(s, L, 0, minus) | (oriented_code(s, L, 1, minus) << 4) | (oriented_code(s, L, 2, minus) << 8);
            if (aa4096[idx] == 'X') d = 1;
        }
    }
    m -= d;
    len32[i] = (int32_t)m;
    out_len[i] = m;
    drop[i] = (int8_t)d;
}

// pass 2: flat over output residues
__global__ void __launch_bounds__(256) k_tr_emit(const uint8_t *__restrict__ in, const int64_t *__restrict__ off, int64_t n_seq,
                                                 int frame, int minus, const int64_t *__restrict__ out_off, const int8_t *__restrict__ drop,
                                                 const uint8_t *__restrict__ aa4096, int64_t total, uint8_t *__restrict__ out) {
    __shared__ __align__(16) uint8_t s_aa[4096];
    reinterpret_cast<uint4 *>(s_aa)[threadIdx.x] = __ldg(reinterpret_cast<const uint4 *>(aa4096) + threadIdx.x);
    __syncthreads();
    const int64_t nchunk = (total + 15) >> 4;
    for (int64_t ch = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; ch < nchunk; ch += (int64_t)gridDim.x * blockDim.x) {
        const int64_t P = ch << 4;
        int64_t i = mg_search_le(out_off, 0, n_seq, P);
        int64_t o_i = __ldg(out_off + i), o_n = __ldg(out_off + i + 1);
        uint32_t w[4] = {0, 0, 0, 0};
        for (int k = 0; k < 16 && P + k < total; k++) {
            const int64_t pos = P + k;
            while (o_n <= pos) { i++; o_i = o_n; o_n = __ldg(out_off + i + 1); }
            const uint8_t *s = in + off[i];
            const int64_t L = off[i + 1] - off[i];
            int lead; int64_t cs, nfull;
            tr_geometry(frame, L, lead, cs, nfull);
            const int64_t a = pos - o_i + drop[i];            // index in the untrimmed translation
            uint32_t aa;
            if (a < lead) aa = 'X';
            else {
                const int64_t q = cs + 3 * (a - lead);
                const uint32_t idx = oriented_code(s, L, q, minus) | (oriented_code(s, L, q + 1, minus) << 4) | (oriented_code(s, L, q + 2, minus) << 8);
                aa = s_aa[idx];
            }
            w[k >> 2] |= aa << ((k & 3) * 8);
        }
        mg_st16(out + P, w[0], w[1], w[2], w[3]);
    }
}

// ---- per-device lazily built translation table ---------------------------------------------------------
static uint8_t *g_aa_table[64] = {nullptr};

static int get_aa_table(int device, uint8_t **out) {
    MG_REQUIRE(device >= 0 && device < 64, "device index out of range");
    if (!g_aa_table[device]) {
        static const char *tcag = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG";
        static const int to_tcag[4] = {2, 1, 3, 0};
        uint8_t t[4096];
        for (int i = 0; i < 4096; i++) {
            const int n0 = i & 15, n1 = (i >> 4) & 15, n2 = (i >> 8) & 15;
            t[i] = (n0 >= 8 || n1 >= 8 || n2 >= 8) ? 'X' : (uint8_t)tcag[to_tcag[n0 & 3] * 16 + to_tcag[n1 & 3] * 4 + to_tcag[n2 & 3]];
        }
        MG_CUDA(cudaMalloc(&g_aa_table[device], 4096));
        MG_CUDA(cudaMemcpy(g_aa_table[device], t, 4096, cudaMemcpyHostToDevice));
    }
    *out = g_aa_table[device];
    return MG_OK;
}

static int check_device(int device) {
    int ndev = 0;
    int rc = mg_device_count(&ndev);
    if (rc) return rc;
    if (device < 0 || device >= ndev) {
        mg_set_error("device %d not available (%d CUDA devices); libmagot_b200 has no CPU fallback", device, ndev);
        return MG_ECUDA;
    }
    return MG_OK;
}

extern "C" int mg_revcomp(int device, const uint8_t *in_host, int64_t n, uint8_t *out_host, void *stream) {
    MG_REQUIRE(n >= 0, "negative length");
    int rc = check_device(device);
    if (rc) return rc;
    if (n == 0) return MG_OK;
    MG_REQUIRE(in_host && out_host, "NULL buffer");
    MG_CUDA(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *d = nullptr;
    const int64_t padded = (n + 15) / 16 * 16;
    MG_CUDA(cudaMallocAsync((void **)&d, 2 * padded, st));
    MG_CUDA(cudaMemcpyAsync(d, in_host, n, cudaMemcpyHostToDevice, st));
    const int blocks = (int)std::min<int64_t>((padded / 16 + 255) / 256, 148 * 16);
    k_revcomp_ascii<<<std::max(blocks, 1), 256, 0, st>>>(d, n, d + padded);
    MG_LAUNCH_CHECK();
    MG_CUDA(cudaMemcpyAsync(out_host, d + padded, n, cudaMemcpyDeviceToHost, st));
    MG_CUDA(cudaStreamSynchronize(st));
    MG_CUDA(cudaFreeAsync(d, st));
    return MG_OK;
}

extern "C" int mg_translate_ascii_table(int device, const uint8_t *codon64, const uint8_t *in_host, const int64_t *off,
                                        int64_t n_seq, int frame, int minus, int trimX, uint8_t *out_host, int64_t out_cap,
                                        int64_t *out_off, int64_t *out_len, void *stream) {
    MG_REQUIRE(n_seq >= 0 && off != nullptr && out_off != nullptr, "bad arguments");
    MG_REQUIRE(frame >= 0 && frame <= 2, "frame must be 0, 1 or 2");
    int rc = check_device(device);
    if (rc) return rc;
    out_off[0] = 0;
    if (n_seq == 0) return MG_OK;
    const int64_t n = off[n_seq] - off[0];
    MG_REQUIRE(off[0] == 0 && n >= 0, "off must start at 0 and be non-decreasing");
    MG_CUDA(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *aa = nullptr;
    if (codon64 == nullptr) {
        rc = get_aa_table(device, &aa);
        if (rc) return rc;
    }
    const int64_t cap = (n + 2) / 3 + n_seq + 16;
    const int64_t scan_tmp = mg_scan_tmp_elems(n_seq) + 2;
    // one arena: in | off | out_off | out_len | len32 | drop | scan tmp | out
    auto al = [](int64_t x) { return (x + 255) / 256 * 256; };
    const int64_t b_in = al(n + 16), b_off = al((n_seq + 1) * 8), b_len = al(n_seq * 8), b_l32 = al(n_seq * 4),
                  b_drop = al(n_seq), b_tmp = al(scan_tmp * 8), b_out = al(cap + 16);
    uint8_t *d = nullptr;
    MG_CUDA(cudaMallocAsync((void **)&d, b_in + 2 * b_off + b_len + b_l32 + b_drop + b_tmp + b_out + 4096, st));
    if (codon64 != nullptr) {                         // caller's codon table (Sequence.translate(library=...), genome.py:795)
        uint8_t t[4096];
        build_aa4096(t, codon64);
        aa = d + b_in + 2 * b_off + b_len + b_l32 + b_drop + b_tmp + b_out;
        MG_CUDA(cudaMemcpyAsync(aa, t, 4096, cudaMemcpyHostToDevice, st));   // pageable source: staged before the call returns
    }
    uint8_t *d_in = d;
    int64_t *d_off = (int64_t *)(d_in + b_in);
    int64_t *d_ooff = (int64_t *)((uint8_t *)d_off + b_off);
    int64_t *d_olen = (int64_t *)((uint8_t *)d_ooff + b_off);
    int32_t *d_l32 = (int32_t *)((uint8_t *)d_olen + b_len);
    int8_t *d_drop = (int8_t *)((uint8_t *)d_l32 + b_l32);
    int64_t *d_tmp = (int64_t *)((uint8_t *)d_drop + b_drop);
    uint8_t *d_out = (uint8_t *)d_tmp + b_tmp;
    if (n) MG_CUDA(cudaMemcpyAsync(d_in, in_host, n, cudaMemcpyHostToDevice, st));
    MG_CUDA(cudaMemcpyAsync(d_off, off, (n_seq + 1) * 8, cudaMemcpyHostToDevice, st));
    k_tr_len<<<(unsigned)((n_seq + 255) / 256), 256, 0, st>>>(d_in, d_off, n_seq, frame, minus, trimX, aa, d_l32, d_olen, d_drop);
    MG_LAUNCH_CHECK();
    rc = mg_scan_i32(d_l32, d_ooff, n_seq, d_tmp, scan_tmp, st);
    if (rc) { cudaFreeAsync(d, st); return rc; }
    MG_CUDA(cudaMemcpyAsync(out_off, d_ooff, (n_seq + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (out_len) MG_CUDA(cudaMemcpyAsync(out_len, d_olen, n_seq * 8, cudaMemcpyDeviceToHost, st));
    MG_CUDA(cudaStreamSynchronize(st));
    const int64_t total = out_off[n_seq];
    if (total > out_cap) {
        cudaFreeAsync(d, st);
        mg_set_error("output buffer too small: need %lld bytes", (long long)total);
        return MG_EINVAL;
    }
    if (total > 0) {
        MG_REQUIRE(out_host != nullptr, "out_host is NULL");
        const int blocks = (int)std::min<int64_t>(((total + 15) / 16 + 255) / 256, 148 * 16);
        k_tr_emit<<<std::max(blocks, 1), 256, 0, st>>>(d_in, d_off, n_seq, frame, minus, d_ooff, d_drop, aa, total, d_out);
        MG_LAUNCH_CHECK();
        MG_CUDA(cudaMemcpyAsync(out_host, d_out, total, cudaMemcpyDeviceToHost, st));
        MG_CUDA(cudaStreamSynchronize(st));
    }
    MG_CUDA(cudaFreeAsync(d, st));
    return MG_OK;
}

extern "C" int mg_translate_ascii(int device, const uint8_t *in_host, const int64_t *off, int64_t n_seq, int frame,
                                  int minus, int trimX, uint8_t *out_host, int64_t out_cap, int64_t *out_off,
                                  int64_t *out_len, void *stream) {
    return mg_translate_ascii_table(device, nullptr, in_host, off, n_seq, frame, minus, trimX, out_host, out_cap, out_off, out_len,
                                    stream);
}
