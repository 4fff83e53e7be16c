// mg_genome.cu -- K0: device-resident nibble-packed genome (replaces the storage half of
// GenomeSequence.__init__, genome.py:856-877) and range decode (GenomeSequence slicing,
// coords2fasta genome_tools.py:656-661, BaseAnnotation.get_seq genome.py:603-608).
#include <algorithm>
#include <numeric>
#include <stdarg.h>
#include <string.h>
#include <thread>
#include "mg_common.cuh"
#include "mg_lookback.cuh"

// ---- error plumbing / misc API -------------------------------------------------------------------
static thread_local char t_err[512] = "";
std::atomic<int64_t> g_mg_launches{0};

void mg_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof(t_err), fmt, ap);
    va_end(ap);
}

extern "C" int mg_version(void) { return MG_VERSION; }
extern "C" const char *mg_last_error(void) { return t_err; }
extern "C" int64_t mg_kernel_launches(void) { return g_mg_launches.load(); }

extern "C" int mg_device_count(int *n_out) {
    MG_REQUIRE(n_out != nullptr, "n_out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *n_out = 0;
        mg_set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return MG_ECUDA;
    }
    *n_out = n;
    return MG_OK;
}

extern "C" int mg_stream_sync(int device, void *stream) {
    MG_CUDA(cudaSetDevice(device));
    MG_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return MG_OK;
}

extern "C" int mg_copy_d2h_async(int device, void *dst_host, const void *src_dev, int64_t n, void *stream) {
    MG_REQUIRE(n >= 0 && (n == 0 || (dst_host && src_dev)), "bad copy arguments");
    MG_CUDA(cudaSetDevice(device));
    if (n > 0) MG_CUDA(cudaMemcpyAsync(dst_host, src_dev, (size_t)n, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return MG_OK;
}

// ---- CUDA graphs: a step (K1 -> K2 -> K3 of one or more plans, on one or several streams) captured once and replayed with a
// single launch.  Nothing in a prepared step waits for the host (mg_plan_prepare_async), so the whole step is capturable; the
// replay removes the per-launch host cost (11 launches per step: at 1/8 of config 4 per GPU the step is ~0.1 ms of kernels).
extern "C" int mg_graph_begin(int device, void *stream) {
    MG_CUDA(cudaSetDevice(device));
    MG_CUDA(cudaStreamBeginCapture((cudaStream_t)stream, cudaStreamCaptureModeThreadLocal));
    return MG_OK;
}

extern "C" int mg_graph_end(int device, void *stream, void **graph_exec_out) {
    MG_REQUIRE(graph_exec_out != nullptr, "graph_exec_out is NULL");
    MG_CUDA(cudaSetDevice(device));
    cudaGraph_t graph = nullptr;
    MG_CUDA(cudaStreamEndCapture((cudaStream_t)stream, &graph));
    cudaGraphExec_t exec = nullptr;
    cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) { mg_set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(e)); return MG_ECUDA; }
    *graph_exec_out = (void *)exec;
    return MG_OK;
}

extern "C" int mg_graph_launch(int device, void *graph_exec, void *stream) {
    MG_REQUIRE(graph_exec != nullptr, "graph_exec is NULL");
    MG_CUDA(cudaSetDevice(device));
    MG_CUDA(cudaGraphLaunch((cudaGraphExec_t)graph_exec, (cudaStream_t)stream));
    return MG_OK;
}

extern "C" int mg_graph_destroy(void *graph_exec) {
    if (graph_exec) cudaGraphExecDestroy((cudaGraphExec_t)graph_exec);
    return MG_OK;
}

// A plan buffer that has to grow is allocated with cudaMallocAsync on the caller's stream.  Inside a capture that becomes a graph
// allocation node that nothing in the graph frees: a second launch of the graph fails, and the plan would keep a pointer with no
// memory behind it until the first replay.  So a call that would grow a buffer while `st` is capturing fails before it queues
// anything; the caller runs the same call once outside the capture, after which the captured call re-uses the buffer.
int mg_refuse_growth_in_capture(cudaStream_t st, const char *what) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    MG_CUDA(cudaStreamIsCapturing(st, &cs));
    if (cs == cudaStreamCaptureStatusNone) return MG_OK;
    mg_set_error("%s would have to grow a plan buffer inside a CUDA graph capture: run it once outside the capture first "
                 "(prepare, and for products emit, with at least the captured capacities)", what);
    return MG_ESTATE;
}

// fork / join helpers for multi-stream steps (also what makes a second stream part of a capture)
extern "C" int mg_stream_wait_stream(int device, void *waiter, void *signaller) {
    MG_CUDA(cudaSetDevice(device));
    cudaEvent_t ev;
    MG_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    cudaError_t e = cudaEventRecord(ev, (cudaStream_t)signaller);
    if (e == cudaSuccess) e = cudaStreamWaitEvent((cudaStream_t)waiter, ev, 0);
    cudaEventDestroy(ev);
    if (e != cudaSuccess) { mg_set_error("stream wait failed: %s", cudaGetErrorString(e)); return MG_ECUDA; }
    return MG_OK;
}

// ---- 4096-entry translation table -----------------------------------------------------------------
// index = n0 | n1<<4 | n2<<8 (n0 = first base of the codon, nibble codes as above).  Any nibble >= 8
// (N, n, '-', IUPAC, exception) gives 'X' (genome.py:816-817); case bit 2 is ignored, which is the
// `.upper()` of genome.py:812.  Amino acids come from codon64[16*b0 + 4*b1 + b2] (A=0 C=1 G=2 T=3), or with
// codon64 == NULL from the reference's table (genome.py:795-802, NCBI table 1).
void build_aa4096(uint8_t *t, const uint8_t *codon64) {
    // reference table is indexed T,C,A,G; our base codes are A=0,C=1,G=2,T=3
    static const char *tcag = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG";
    static const int to_tcag[4] = {2, 1, 3, 0};
    for (int i = 0; i < 4096; i++) {
        const int n0 = i & 15, n1 = (i >> 4) & 15, n2 = (i >> 8) & 15;
        if (n0 >= 8 || n1 >= 8 || n2 >= 8) {
            t[i] = 'X';
        } else if (codon64) {
            t[i] = codon64[(n0 & 3) * 16 + (n1 & 3) * 4 + (n2 & 3)];
        } else {
            t[i] = (uint8_t)tcag[to_tcag[n0 & 3] * 16 + to_tcag[n1 & 3] * 4 + to_tcag[n2 & 3]];
        }
    }
}

// ---- create / destroy -----------------------------------------------------------------------------
extern "C" int mg_genome_create(int device, int64_t n_contigs, const int64_t *contig_len, mg_genome **out) {
    MG_REQUIRE(out != nullptr, "out is NULL");
    MG_REQUIRE(n_contigs >= 0 && (n_contigs == 0 || contig_len != nullptr), "bad contig table");
    int ndev = 0;
    int rc = mg_device_count(&ndev);
    if (rc != MG_OK) return rc;
    if (device < 0 || device >= ndev) {
        mg_set_error("device %d not available (%d CUDA devices); libmagot_b200 has no CPU fallback", device, ndev);
        return MG_ECUDA;
    }
    MG_CUDA(cudaSetDevice(device));
    mg_genome *g = new mg_genome();
    g->device = device;
    g->n_contigs = n_contigs;
    g->h_contig_len.assign(contig_len, contig_len + n_contigs);
    g->h_contig_base.resize(n_contigs + 1);
    int64_t base = MG_FRONT_PAD;
    for (int64_t c = 0; c < n_contigs; c++) {
        if (contig_len[c] < 0) { delete g; mg_set_error("negative contig length"); return MG_EINVAL; }
        g->h_contig_base[c] = base;
        base += (contig_len[c] + 31) / 32 * 32;
    }
    g->h_contig_base[n_contigs] = base;
    g->total_bases = base;
    const int64_t words = 2 * base / 8 + MG_TAIL_WORDS;           // forward plane + reverse-complement plane
    MG_CUDA(cudaMalloc(&g->d_packed, words * sizeof(uint32_t)));
    // padding decodes as 'N' (0x8 per nibble) so that stray reads are harmless and deterministic
    MG_CUDA(cudaMemset(g->d_packed, 0x88, words * sizeof(uint32_t)));
    MG_CUDA(cudaMalloc(&g->d_contig_len, std::max<int64_t>(1, n_contigs) * sizeof(int64_t)));
    MG_CUDA(cudaMalloc(&g->d_contig_base, (n_contigs + 1) * sizeof(int64_t)));
    if (n_contigs) MG_CUDA(cudaMemcpy(g->d_contig_len, contig_len, n_contigs * sizeof(int64_t), cudaMemcpyHostToDevice));
    MG_CUDA(cudaMemcpy(g->d_contig_base, g->h_contig_base.data(), (n_contigs + 1) * sizeof(int64_t), cudaMemcpyHostToDevice));
    MG_CUDA(cudaMalloc(&g->d_exc_count, sizeof(unsigned long long)));
    g->exc_cap = 1 << 16;
    MG_CUDA(cudaMalloc(&g->d_exc_pos, g->exc_cap * sizeof(int64_t)));
    MG_CUDA(cudaMalloc(&g->d_exc_byte, g->exc_cap));
    uint8_t tbl[4096];
    build_aa4096(tbl, nullptr);
    MG_CUDA(cudaMalloc(&g->d_aa4096, 4096));
    MG_CUDA(cudaMemcpy(g->d_aa4096, tbl, 4096, cudaMemcpyHostToDevice));
    uint8_t tblh[4096];
    for (uint32_t c = 0; c < 4096; c++) tblh[mg_aa_slot(c)] = tbl[c];
    MG_CUDA(cudaMalloc(&g->d_aa4096h, 4096));
    MG_CUDA(cudaMemcpy(g->d_aa4096h, tblh, 4096, cudaMemcpyHostToDevice));
    g->device_bytes = words * 4 + (2 * n_contigs + 1) * 8 + 4096;
    // keep freed stream-ordered allocations cached: plans are created and destroyed per batch
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    *out = g;
    return MG_OK;
}

void mg_sixframe_free(mg_genome *g);

extern "C" int mg_genome_destroy(mg_genome *g) {
    if (!g) return MG_OK;
    cudaSetDevice(g->device);
    mg_sixframe_free(g);
    cudaFree(g->d_packed);
    cudaFree(g->d_contig_len);
    cudaFree(g->d_contig_base);
    cudaFree(g->d_exc_pos);
    cudaFree(g->d_exc_byte);
    cudaFree(g->d_exc_count);
    cudaFree(g->d_stage);
    cudaFree(g->d_raw);
    cudaFree(g->d_strip_tmp);
    cudaFree(g->d_aa4096);
    cudaFree(g->d_aa4096h);
    cudaFree(g->d_stops);
    cudaFree(g->d_stops_alt);
    if (g->h_pin) cudaFreeHost(g->h_pin);
    delete g;
    return MG_OK;
}

extern "C" int64_t mg_genome_bytes(const mg_genome *g) { return g ? g->device_bytes : 0; }

int mg_ensure_stage(mg_genome *g, int64_t bytes) {
    if (g->stage_cap >= bytes) return MG_OK;
    if (g->d_stage) MG_CUDA(cudaFree(g->d_stage));
    g->d_stage = nullptr;
    g->stage_cap = 0;
    MG_CUDA(cudaMalloc(&g->d_stage, bytes));
    g->stage_cap = bytes;
    return MG_OK;
}

int mg_ensure_pin(mg_genome *g, int64_t bytes) {
    if (g->pin_cap >= bytes) return MG_OK;
    if (g->h_pin) MG_CUDA(cudaFreeHost(g->h_pin));
    g->h_pin = nullptr;
    g->pin_cap = 0;
    MG_CUDA(cudaMallocHost(&g->h_pin, bytes));
    g->pin_cap = bytes;
    return MG_OK;
}

// ---- K0 pack kernel ---------------------------------------------------------------------------------
// One thread packs 16 ASCII bytes (one 16-byte load) into 2 words (one 8-byte store).  HBM traffic:
// 1 B/base read + 0.5 B/base written.  Bytes outside the 15-symbol alphabet become code 15 and are
// appended to the exception list (rare in real assemblies; dense lists still work, only slower).
__global__ void __launch_bounds__(256) k_pack(const uint8_t *__restrict__ ascii, int64_t n, int64_t g0, int64_t two_T,
                                              uint32_t *__restrict__ packed, int64_t *__restrict__ exc_pos,
                                              uint8_t *__restrict__ exc_byte, int64_t exc_cap,
                                              unsigned long long *__restrict__ exc_count) {
    const int64_t nchunk = (n + 15) >> 4;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nchunk; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b0 = i << 4;
        uint32_t w[4];
        if (b0 + 16 <= n) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(ascii + b0));
            w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
        } else {
            w[0] = w[1] = w[2] = w[3] = 0x4E4E4E4Eu;   // 'N' padding past the end of the chunk
            for (int k = 0; b0 + k < n; k++) {
                const uint32_t c = ascii[b0 + k];
                w[k >> 2] = (w[k >> 2] & ~(0xFFu << ((k & 3) * 8))) | (c << ((k & 3) * 8));
            }
        }
        uint32_t o[2] = {0u, 0u};
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const uint8_t c = (uint8_t)(w[k >> 2] >> ((k & 3) * 8));
            const uint32_t code = mg_encode(c);
            o[k >> 3] |= code << ((k & 7) * 4);
            if (code == MG_CODE_EXC && b0 + k < n) {
                const unsigned long long slot = atomicAdd(exc_count, 1ull);
                if ((int64_t)slot < exc_cap) {
                    exc_pos[slot] = g0 + b0 + k;
                    exc_byte[slot] = c;
                }
            }
        }
        *reinterpret_cast<uint2 *>(packed + ((g0 + b0) >> 3)) = make_uint2(o[0], o[1]);
        // reverse-complement plane: forward bases [G, G+16) are bases [2T-16-G, 2T-G) of the second plane
        const uint64_t rc = mg_rc_nib16(((uint64_t)o[1] << 32) | o[0]);
        *reinterpret_cast<uint2 *>(packed + ((two_T - 16 - (g0 + b0)) >> 3)) = make_uint2((uint32_t)rc, (uint32_t)(rc >> 32));
    }
}

static int pack_device_chunk(mg_genome *g, int64_t gbase, const uint8_t *d_ascii, int64_t n, cudaStream_t st) {
    for (;;) {
        MG_CUDA(cudaMemsetAsync(g->d_exc_count, 0, sizeof(unsigned long long), st));
        const int64_t nchunk = (n + 15) / 16;
        const int blocks = (int)std::min<int64_t>((nchunk + 255) / 256, 148 * 16);
        k_pack<<<std::max(blocks, 1), 256, 0, st>>>(d_ascii, n, gbase, 2 * g->total_bases, g->d_packed, g->d_exc_pos, g->d_exc_byte,
                                                   g->exc_cap, g->d_exc_count);
        MG_LAUNCH_CHECK();
        unsigned long long cnt = 0;
        MG_CUDA(cudaMemcpyAsync(&cnt, g->d_exc_count, sizeof(cnt), cudaMemcpyDeviceToHost, st));
        MG_CUDA(cudaStreamSynchronize(st));
        if ((int64_t)cnt > g->exc_cap) {              // rare: grow and redo this chunk
            MG_CUDA(cudaFree(g->d_exc_pos));
            MG_CUDA(cudaFree(g->d_exc_byte));
            g->exc_cap = (int64_t)cnt + 1024;
            MG_CUDA(cudaMalloc(&g->d_exc_pos, g->exc_cap * sizeof(int64_t)));
            MG_CUDA(cudaMalloc(&g->d_exc_byte, g->exc_cap));
            continue;
        }
        if (cnt) {
            const size_t old = g->h_exc_pos.size();
            g->h_exc_pos.resize(old + cnt);
            g->h_exc_byte.resize(old + cnt);
            MG_CUDA(cudaMemcpy(g->h_exc_pos.data() + old, g->d_exc_pos, cnt * sizeof(int64_t), cudaMemcpyDeviceToHost));
            MG_CUDA(cudaMemcpy(g->h_exc_byte.data() + old, g->d_exc_byte, cnt, cudaMemcpyDeviceToHost));
        }
        return MG_OK;
    }
}

static int check_pack_args(mg_genome *g, int64_t contig, int64_t offset, const void *p, int64_t n) {
    MG_REQUIRE(g != nullptr, "genome handle is NULL");
    MG_REQUIRE(contig >= 0 && contig < g->n_contigs, "contig index out of range");
    MG_REQUIRE(n >= 0 && offset >= 0 && offset + n <= g->h_contig_len[contig], "chunk outside the contig");
    MG_REQUIRE(n == 0 || p != nullptr, "ascii is NULL");
    MG_REQUIRE(offset % 32 == 0, "chunk offset must be a multiple of 32 bases");
    MG_REQUIRE(n % 32 == 0 || offset + n == g->h_contig_len[contig], "chunk length must be a multiple of 32 unless it ends the contig");
    return MG_OK;
}

extern "C" int mg_genome_pack_device(mg_genome *g, int64_t contig, int64_t offset, const uint8_t *ascii_dev,
                                     int64_t n, void *stream) {
    int rc = check_pack_args(g, contig, offset, ascii_dev, n);
    if (rc) return rc;
    MG_REQUIRE(((uintptr_t)ascii_dev & 15) == 0, "device text must be 16-byte aligned");
    MG_CUDA(cudaSetDevice(g->device));
    g->finalized = false;
    g->generation++;
    g->stops_valid = g->stops_alt_valid = false;
    if (n == 0) return MG_OK;
    return pack_device_chunk(g, g->h_contig_base[contig] + offset, ascii_dev, n, (cudaStream_t)stream);
}

extern "C" int mg_genome_pack(mg_genome *g, int64_t contig, int64_t offset, const uint8_t *ascii, int64_t n, void *stream) {
    int rc = check_pack_args(g, contig, offset, ascii, n);
    if (rc) return rc;
    MG_CUDA(cudaSetDevice(g->device));
    g->finalized = false;
    g->generation++;
    g->stops_valid = g->stops_alt_valid = false;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t STAGE = 64ll << 20;
    rc = mg_ensure_stage(g, std::min<int64_t>(STAGE, (n + 255) / 256 * 256));
    if (rc) return rc;
    for (int64_t done = 0; done < n;) {
        const int64_t m = std::min<int64_t>(g->stage_cap / 32 * 32, n - done);
        MG_CUDA(cudaMemcpyAsync(g->d_stage, ascii + done, m, cudaMemcpyHostToDevice, st));
        rc = pack_device_chunk(g, g->h_contig_base[contig] + offset + done, g->d_stage, m, st);
        if (rc) return rc;
        done += m;
    }
    return MG_OK;
}

// ---- K0f: FASTA body -> ASCII without line ends, on the device ----------------------------------------------------------
// Replaces `seq = seq + line.replace('\n','').replace('\r','')` (genome.py:875) for a whole record body: a stream compaction
// that drops every CR / LF byte and keeps everything else (spaces, case, any byte: the reference keeps them too).
// One tile = 256 threads x 16 raw bytes.  Kept bytes are ranked with a warp/block scan, the tile's base comes from the
// decoupled look-back (single pass, tiles in ticket order), the tile's survivors are staged in shared memory and written
// as one contiguous run.  HBM: 1 B read + <= 1 B written per raw byte; the host never touches the sequence bytes.
#define STRIP_THREADS 256
#define STRIP_TILE (STRIP_THREADS * 16)
__global__ void __launch_bounds__(STRIP_THREADS) k_fasta_strip(const uint8_t *__restrict__ raw, int64_t n, unsigned long long *tmp,
                                                                uint8_t *__restrict__ dst, int64_t *__restrict__ kept_total) {
    __shared__ int64_t s_warp[STRIP_THREADS / 32];
    __shared__ int64_t s_prefix;
    __shared__ unsigned int s_tile;
    __shared__ uint8_t s_out[STRIP_TILE];
    const int64_t tile = mg_next_tile(tmp, &s_tile);
    const int64_t b0 = tile * STRIP_TILE + (int64_t)threadIdx.x * 16;
    uint32_t w[4];
    if (b0 + 16 <= n) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(raw + b0));
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    } else {
        w[0] = w[1] = w[2] = w[3] = 0x0A0A0A0Au;       // past the end: line feeds, i.e. dropped
        for (int k = 0; b0 + k < n; k++) {
            const uint32_t c = raw[b0 + k];
            w[k >> 2] = (w[k >> 2] & ~(0xFFu << ((k & 3) * 8))) | (c << ((k & 3) * 8));
        }
    }
    uint32_t keep = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const uint32_t c = (w[k >> 2] >> ((k & 3) * 8)) & 0xFFu;
        keep |= (uint32_t)(c != 0x0Au && c != 0x0Du) << k;
    }
    const int cnt = __popc(keep);
    int64_t total;
    const int64_t incl = mg_block_incl_scan((int64_t)cnt, s_warp, &total);
    const int64_t prefix = mg_lookback(tmp, tile, total, &s_prefix);
    int pos = (int)(incl - cnt);
#pragma unroll
    for (int k = 0; k < 16; k++) {
        if ((keep >> k) & 1u) s_out[pos++] = (uint8_t)(w[k >> 2] >> ((k & 3) * 8));
    }
    __syncthreads();
    for (int i = threadIdx.x; i < (int)total; i += STRIP_THREADS) dst[prefix + i] = s_out[i];
    if (tile == gridDim.x - 1 && threadIdx.x == 0) *kept_total = prefix + total;
}

// Host side of K0f: the caller's FASTA bytes are pageable; a pageable cudaMemcpy runs at ~10 GB/s (the round-1 ingest rate).
// Worker threads copy the NEXT trip into one of two page-locked buffers while the device takes the previous trip from the
// other buffer at the PCIe rate and strips it; the number of bases the strip kept comes back in a page-locked word that the
// host reads after its own copy, i.e. without ever waiting for it.
void mg_parallel_copy(const uint8_t *src, uint8_t *dst, int64_t n) {
    int T = (int)std::thread::hardware_concurrency();
    T = std::max(1, std::min(T, 8));
    if (n < (4 << 20)) T = 1;
    std::vector<std::thread> th;
    const int64_t per = ((n + T - 1) / T + 4095) / 4096 * 4096;
    for (int t = 1; t < T; t++) {
        const int64_t a = std::min(n, t * per), b = std::min(n, a + per);
        if (b > a) th.emplace_back([=]() { memcpy(dst + a, src + a, (size_t)(b - a)); });
    }
    memcpy(dst, src, (size_t)std::min(n, per));
    for (auto &x : th) x.join();
}

// Line-end bytes (CR, LF) inside each of n_ranges byte ranges [lo, hi) of a FASTA text: body length of a record = its bytes
// minus these (genome.py:875 drops exactly '\n' and '\r').  Host only; the ranges are shared out over up to 8 threads by bytes.
extern "C" int mg_count_line_ends(const uint8_t *data, int64_t n, int64_t n_ranges, const int64_t *lo, const int64_t *hi, int64_t *out) {
    MG_REQUIRE((data || n == 0) && n_ranges >= 0 && (n_ranges == 0 || (lo && hi && out)), "bad arguments");
    for (int64_t r = 0; r < n_ranges; r++) MG_REQUIRE(lo[r] >= 0 && hi[r] >= lo[r] && hi[r] <= n, "range outside the text");
    int T = (int)std::thread::hardware_concurrency();
    T = std::max(1, std::min(T, 8));
    if (n < (8 << 20)) T = 1;
    auto work = [&](int64_t r0, int64_t r1) {
        for (int64_t r = r0; r < r1; r++) {
            const uint8_t *p = data + lo[r];
            const int64_t m = hi[r] - lo[r];
            int64_t c = 0;
            for (int64_t i = 0; i < m; i += 1 << 16) {    // blocks small enough for a byte-wide vectorised count
                const int64_t e = std::min<int64_t>(m, i + (1 << 16));
                uint32_t cc = 0;
                for (int64_t j = i; j < e; j++) cc += (uint32_t)((p[j] == '\n') | (p[j] == '\r'));
                c += cc;
            }
            out[r] = c;
        }
    };
    std::vector<std::thread> th;
    int64_t r0 = 0, acc = 0;
    const int64_t per = n / T + 1;
    for (int64_t r = 0; r < n_ranges; r++) {
        acc += hi[r] - lo[r];
        if (acc >= per && (int)th.size() < T - 1) { th.emplace_back(work, r0, r + 1); r0 = r + 1; acc = 0; }
    }
    work(r0, n_ranges);
    for (auto &x : th) x.join();
    return MG_OK;
}

extern "C" int mg_genome_pack_fasta(mg_genome *g, int64_t contig, const uint8_t *raw, int64_t n_raw, void *stream) {
    MG_REQUIRE(g != nullptr, "genome handle is NULL");
    MG_REQUIRE(contig >= 0 && contig < g->n_contigs, "contig index out of range");
    MG_REQUIRE(n_raw >= 0 && (n_raw == 0 || raw != nullptr), "bad FASTA body");
    MG_CUDA(cudaSetDevice(g->device));
    g->finalized = false;
    g->generation++;
    g->stops_valid = g->stops_alt_valid = false;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t RAW = 64ll << 20;                   // raw bytes per trip (multiple of the tile)
    const int64_t clen = g->h_contig_len[contig];
    // one size for the life of the handle (a FASTA with thousands of scaffolds must not re-allocate page-locked memory per
    // scaffold): what the longest contig needs with 60-column lines, at most one trip
    int64_t longest = 0;
    for (int64_t L : g->h_contig_len) longest = std::max(longest, L);
    const int64_t want_cap = std::min<int64_t>(RAW, ((longest + longest / 16 + 4096) + STRIP_TILE - 1) / STRIP_TILE * STRIP_TILE);
    const int64_t chunk_cap = std::max(want_cap, std::min<int64_t>(RAW, (n_raw + STRIP_TILE - 1) / STRIP_TILE * STRIP_TILE));
    if (g->raw_cap < chunk_cap) {
        if (g->d_raw) MG_CUDA(cudaFree(g->d_raw));
        if (g->d_strip_tmp) MG_CUDA(cudaFree(g->d_strip_tmp));
        g->d_raw = nullptr; g->d_strip_tmp = nullptr; g->raw_cap = 0;
        MG_CUDA(cudaMalloc(&g->d_raw, chunk_cap));
        MG_CUDA(cudaMalloc(&g->d_strip_tmp, (chunk_cap / STRIP_TILE + 4) * sizeof(unsigned long long)));
        g->raw_cap = chunk_cap;
    }
    int rc = mg_ensure_stage(g, chunk_cap + 256);     // ASCII staging: up to 31 carried bytes + one stripped chunk
    if (rc) return rc;
    rc = mg_ensure_pin(g, 2 * g->raw_cap + 64);       // two page-locked trip buffers + the kept-bytes word
    if (rc) return rc;
    uint8_t *pin[2] = {g->h_pin, g->h_pin + g->raw_cap};
    volatile int64_t *h_kept = reinterpret_cast<volatile int64_t *>(g->h_pin + 2 * g->raw_cap);
    int64_t *d_kept = reinterpret_cast<int64_t *>(g->d_strip_tmp + (g->raw_cap / STRIP_TILE + 2));
    int64_t carry = 0, done_bases = 0;
    int64_t m_next = std::min<int64_t>(g->raw_cap, n_raw);
    if (m_next > 0) mg_parallel_copy(raw, pin[0], m_next);
    int k = 0;
    for (int64_t done = 0; done < n_raw || (n_raw == 0 && done == 0); k++) {
        const int64_t m = m_next;
        if (m > 0) {
            const int64_t nt = (m + STRIP_TILE - 1) / STRIP_TILE;
            MG_CUDA(cudaMemcpyAsync(g->d_raw, pin[k & 1], m, cudaMemcpyHostToDevice, st));
            MG_CUDA(cudaMemsetAsync(g->d_strip_tmp, 0, (nt + 1) * sizeof(unsigned long long), st));
            k_fasta_strip<<<(unsigned)nt, STRIP_THREADS, 0, st>>>(g->d_raw, m, g->d_strip_tmp, g->d_stage + carry, d_kept);
            MG_LAUNCH_CHECK();
            MG_CUDA(cudaMemcpyAsync((void *)h_kept, d_kept, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        }
        done += m;
        const bool last = done >= n_raw;
        // the next trip is copied by the host while the device copies / strips this one; its buffer was last read by the trip
        // before this one, whose pack has been waited for
        m_next = last ? 0 : std::min<int64_t>(g->raw_cap, n_raw - done);
        if (m_next > 0) mg_parallel_copy(raw + done, pin[(k + 1) & 1], m_next);
        int64_t kept = 0;
        if (m > 0) { MG_CUDA(cudaStreamSynchronize(st)); kept = *h_kept; }
        const int64_t avail = carry + kept;
        const int64_t npack = last ? avail : avail / 32 * 32;
        if (done_bases + npack > clen || (last && done_bases + npack != clen)) {
            cudaStreamSynchronize(st);
            mg_set_error("FASTA body of contig %lld holds %s%lld bases, the genome was created with %lld", (long long)contig,
                         last ? "" : "more than ", (long long)(done_bases + npack), (long long)clen);
            return MG_EINVAL;
        }
        if (npack > 0) {
            rc = pack_device_chunk(g, g->h_contig_base[contig] + done_bases, g->d_stage, npack, st);
            if (rc) return rc;
        }
        carry = avail - npack;
        if (carry > 0 && npack > 0) MG_CUDA(cudaMemcpyAsync(g->d_stage, g->d_stage + npack, carry, cudaMemcpyDeviceToDevice, st));
        done_bases += npack;
        if (n_raw == 0) break;
    }
    return MG_OK;
}

extern "C" int mg_genome_finalize(mg_genome *g, int64_t *n_exceptions_out) {
    MG_REQUIRE(g != nullptr, "genome handle is NULL");
    MG_CUDA(cudaSetDevice(g->device));
    const int64_t n = (int64_t)g->h_exc_pos.size();
    // a position packed twice (re-sent chunk) keeps its last byte
    std::vector<int64_t> idx(n);
    std::iota(idx.begin(), idx.end(), 0);
    std::stable_sort(idx.begin(), idx.end(), [&](int64_t a, int64_t b) { return g->h_exc_pos[a] < g->h_exc_pos[b]; });
    std::vector<int64_t> pos;
    std::vector<uint8_t> byt;
    pos.reserve(n);
    byt.reserve(n);
    for (int64_t k = 0; k < n; k++) {
        const int64_t i = idx[k];
        if (!pos.empty() && pos.back() == g->h_exc_pos[i]) byt.back() = g->h_exc_byte[i];
        else { pos.push_back(g->h_exc_pos[i]); byt.push_back(g->h_exc_byte[i]); }
    }
    g->n_exc = (int64_t)pos.size();
    if (g->n_exc > g->exc_cap) {
        MG_CUDA(cudaFree(g->d_exc_pos));
        MG_CUDA(cudaFree(g->d_exc_byte));
        g->exc_cap = g->n_exc;
        MG_CUDA(cudaMalloc(&g->d_exc_pos, g->exc_cap * sizeof(int64_t)));
        MG_CUDA(cudaMalloc(&g->d_exc_byte, g->exc_cap));
    }
    if (g->n_exc) {
        MG_CUDA(cudaMemcpy(g->d_exc_pos, pos.data(), g->n_exc * sizeof(int64_t), cudaMemcpyHostToDevice));
        MG_CUDA(cudaMemcpy(g->d_exc_byte, byt.data(), g->n_exc, cudaMemcpyHostToDevice));
    }
    g->h_exc_pos.swap(pos);
    g->h_exc_byte.swap(byt);
    g->finalized = true;
    g->generation++;
    g->stops_valid = g->stops_alt_valid = false;
    if (n_exceptions_out) *n_exceptions_out = g->n_exc;
    return MG_OK;
}

// ---- range decode -----------------------------------------------------------------------------------
// out[i] for i in [0, n) = base g_lo+i of whichever plane g_lo points into.  16 bytes / thread.
__global__ void __launch_bounds__(256) k_fetch(const uint32_t *__restrict__ packed, int64_t g_lo, int64_t n, int minus,
                                               const int64_t *__restrict__ exc_pos, const uint8_t *__restrict__ exc_byte,
                                               int64_t n_exc, uint8_t *__restrict__ out) {
    const int64_t nchunk = (n + 15) >> 4;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nchunk; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o = i << 4;
        const uint64_t v = mg_ld_nib16(packed, g_lo + o);       // g_lo already points into the right plane
        uint32_t b0, b1, b2, b3;
        mg_decode8((uint32_t)v, b0, b1);
        mg_decode8((uint32_t)(v >> 32), b2, b3);
        if (!minus && n_exc > 0) {
            uint32_t w[4] = {b0, b1, b2, b3};
            for (int k = 0; k < 16; k++) {
                if (((v >> (4 * k)) & 15u) == MG_CODE_EXC && o + k < n) {
                    const uint32_t c = mg_exc_byte(exc_pos, exc_byte, n_exc, g_lo + o + k);
                    w[k >> 2] = (w[k >> 2] & ~(0xFFu << ((k & 3) * 8))) | (c << ((k & 3) * 8));
                }
            }
            b0 = w[0]; b1 = w[1]; b2 = w[2]; b3 = w[3];
        }
        mg_st16(out + o, b0, b1, b2, b3);
    }
}

extern "C" int mg_genome_fetch(mg_genome *g, int64_t contig, int64_t lo, int64_t hi, int minus, uint8_t *out_host, void *stream) {
    MG_REQUIRE(g != nullptr, "genome handle is NULL");
    MG_REQUIRE(g->finalized, "mg_genome_finalize has not been called");
    MG_REQUIRE(contig >= 0 && contig < g->n_contigs, "contig index out of range");
    MG_REQUIRE(lo >= 0 && lo <= hi && hi <= g->h_contig_len[contig], "range outside the contig");
    if (hi == lo) return MG_OK;
    MG_REQUIRE(out_host != nullptr, "out_host is NULL");
    MG_CUDA(cudaSetDevice(g->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = hi - lo;
    const int64_t STAGE = 64ll << 20;
    int rc = mg_ensure_stage(g, std::min<int64_t>(STAGE, (n + 255) / 256 * 256));
    if (rc) return rc;
    const int64_t gl = g->h_contig_base[contig] + lo;
    const int64_t step = g->stage_cap / 16 * 16;
    for (int64_t done = 0; done < n;) {
        const int64_t m = std::min<int64_t>(step, n - done);
        // forward: output [done, done+m) = bases gl+done ..; minus: output [done, done+m) = rc of bases [gl+n-done-m, gl+n-done)
        // minus: output byte i is the complement of base gl+n-1-i, i.e. base (2T - gl - n) + i of the reverse plane
        const int64_t sub_lo = minus ? 2 * g->total_bases - gl - n + done : gl + done;
        const int blocks = (int)std::min<int64_t>(((m + 15) / 16 + 255) / 256, 148 * 16);
        k_fetch<<<std::max(blocks, 1), 256, 0, st>>>(g->d_packed, sub_lo, m, minus, g->d_exc_pos, g->d_exc_byte, g->n_exc, g->d_stage);
        MG_LAUNCH_CHECK();
        MG_CUDA(cudaMemcpyAsync(out_host + done, g->d_stage, m, cudaMemcpyDeviceToHost, st));
        MG_CUDA(cudaStreamSynchronize(st));
        done += m;
    }
    return MG_OK;
}
