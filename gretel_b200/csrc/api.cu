// C-ABI plumbing of libhanselx.so: lifetime, ingestion entry points, the scalar Hansel
// surface and bulk matrix I/O.  See include/hanselx.h for the reference interface each
// function replaces.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include <atomic>

#include "hx_internal.cuh"
#include "scan.cuh"

static thread_local char g_err[512] = "";

void hx_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static void release_counts(hx_matrix *h) {
    for (int g = 0; g < HX_MAX_PEERS; ++g) {
        if (h->ipc_opened[g]) cudaIpcCloseMemHandle(h->ipc_opened[g]);
        h->ipc_opened[g] = nullptr;
        h->peer_host[g] = nullptr;
    }
    h->peer_world = 0;
    if (h->cnt) {
        if (h->cnt_ipc) { cudaStreamSynchronize(h->stream); cudaFree(h->cnt); }
        else cudaFreeAsync(h->cnt, h->stream);
    }
    h->cnt = nullptr;
    h->cnt_ipc = false;
    h->cnt_elems = 0;
}

HxCnt hx_cnt_ref(const hx_matrix *h) {
    HxCnt c;
    c.local = h->cnt;
    c.peer = h->d_peer_tbl;
    c.world = h->peer_world > 1 ? h->peer_world : 1;
    c.rows_per = h->peer_world > 1 ? h->peer_rows_per : 1;
    return c;
}

namespace {

__global__ void k_fold_counts(const uint32_t *__restrict__ cnt, float *__restrict__ band, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const uint32_t c = cnt[i];
        if (c) band[i] += (float)c;
    }
}

__global__ void k_add_one(float *p, float amount) { *p += amount; }

// counts (16-byte aligned allocation, size in bytes), totals[8] and the error word in one launch
__global__ void k_reset_counts(uint4 *__restrict__ cnt, size_t bytes, unsigned long long *__restrict__ totals,
                               int *__restrict__ err) {
    const size_t n16 = bytes / 16;
    const uint4 z = make_uint4(0, 0, 0, 0);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) cnt[i] = z;
    if (blockIdx.x == 0) {
        uint8_t *tail = reinterpret_cast<uint8_t *>(cnt) + n16 * 16;
        for (size_t i = threadIdx.x; i < bytes - n16 * 16; i += blockDim.x) tail[i] = 0;
        if (threadIdx.x < 8) totals[threadIdx.x] = 0;
        if (threadIdx.x == 8) *err = 0;
    }
}

// ---- packed exchange: the 49 uint32 counts of a site pair travel as 49 x uint16 in 25 words.  Summing the
// words as uint32 across GPUs is exact as long as no 16-bit lane carries, i.e. every count <= 65535/world on
// every rank; the pack kernel raises a flag word otherwise and the caller falls back to the plain exchange.
#define HX_PACK_WORDS 25
__global__ void k_pack_counts(const uint32_t *__restrict__ cnt, int64_t n_pairs, uint32_t lim16,
                              uint32_t *__restrict__ packed, int64_t flag_at) {
    // one thread per packed word: words of consecutive threads are consecutive in memory
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs * HX_PACK_WORDS) return;
    const int64_t p = i / HX_PACK_WORDS;
    const int w = (int)(i - p * HX_PACK_WORDS);
    const uint32_t *c = cnt + p * HX_CELL + 2 * w;
    const uint32_t lo = c[0], hi = 2 * w + 1 < HX_CELL ? c[1] : 0u;
    if (lo > lim16 || hi > lim16) packed[flag_at] = 1u;
    packed[i] = (lo & 0xffffu) | (hi << 16);
}

__global__ void k_unpack_counts(const uint32_t *__restrict__ packed, int64_t n_pairs, uint32_t *__restrict__ cnt,
                                int64_t flag_at) {
    if (packed[flag_at] != 0u) return;                                 // some rank overflowed: leave the partials
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs * HX_PACK_WORDS) return;
    const int64_t p = i / HX_PACK_WORDS;
    const int w = (int)(i - p * HX_PACK_WORDS);
    const uint32_t v = packed[i];
    uint32_t *c = cnt + p * HX_CELL + 2 * w;
    c[0] = v & 0xffffu;
    if (2 * w + 1 < HX_CELL) c[1] = v >> 16;
}

// compact wire format -> the packed arrays the ingestion kernels read
__global__ void k_widen_klen(const uint16_t *__restrict__ klen, int64_t n, int64_t *__restrict__ out /* n+1 */) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) out[i] = i < n ? (int64_t)klen[i] : 0;
}

__global__ void k_unpack_nibbles(const uint32_t *__restrict__ in, int64_t n_words, uint2 *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words) return;
    const uint32_t w = in[i];                    // 4 bytes = 8 codes, low nibble first
    uint2 o;
    o.x = (w & 0xfu) | ((w >> 4 & 0xfu) << 8) | ((w >> 8 & 0xfu) << 16) | ((w >> 12 & 0xfu) << 24);
    o.y = (w >> 16 & 0xfu) | ((w >> 20 & 0xfu) << 8) | ((w >> 24 & 0xfu) << 16) | ((w >> 28 & 0xfu) << 24);
    out[i] = o;
}

__global__ void k_reweight_one(float *p, double ratio, double *removed) {
    const double old = (double)*p;
    const double nw = old - (ratio * old);
    *p = (float)nw;
    *removed = old - nw;
}

int in_band(const hx_matrix *h, int a, int b, int64_t i, int64_t j) {
    if (a < 0 || a >= HX_NSYM || b < 0 || b >= HX_NSYM) return HX_E_ARG;
    if (i < 0 || j < 0 || i > (int64_t)h->N + 1 || j > (int64_t)h->N + 1) return HX_E_ARG;
    if (j - i < 1 || j - i > h->W) return HX_E_BAND;
    return HX_OK;
}

void free_all(hx_matrix *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    hx_lr_free(h);
    hx_l2_free(h);
    hx_wire_free(h);
    hx_support_free(h);
    hx_score_free(h);
    if (h->d_peer_tbl) cudaFree(h->d_peer_tbl);
    cudaStream_t st = h->stream;
    h->band.release(st);
    release_counts(h);
    h->d_totals.release(st); h->d_err.release(st);
    h->s_rank.release(st); h->s_off.release(st); h->s_codes.release(st);
    h->s_klen.release(st); h->s_codes4.release(st); h->s_scan.release(st);
    h->scnt.release(st); h->vseen.release(st); h->d_path.release(st); h->d_stats.release(st); h->d_site.release(st);
    h->terms.release(st); h->logm.release(st); h->termsq.release(st); h->logmq.release(st);
    h->spec.release(st); h->guess.release(st); h->spec_ok.release(st); h->cand_idx.release(st);
    h->d_partials.release(st); h->d_flags.release(st);
    h->d_run_end.release(st); h->d_run_list.release(st); h->d_jobs.release(st); h->d_misc.release(st);
    h->d_pack.release(st);
    if (st) cudaStreamSynchronize(st);
    free(h->h_pinned);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->host_ev) cudaEventDestroy(h->host_ev);
    if (h->sum_stream) { cudaStreamSynchronize(h->sum_stream); cudaStreamDestroy(h->sum_stream); }
    for (int b = 0; b < 2; ++b) if (h->sum_done[b]) cudaEventDestroy(h->sum_done[b]);
    if (h->site_ready) cudaEventDestroy(h->site_ready);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    free(h);
}

}  // namespace

extern "C" {

const char *hx_last_error(void) { return g_err; }
int hx_version(void) { return 100; }

int hx_device_count(int *n) {
    HX_CHECK_ARG(n);
    HX_CUDA(cudaGetDeviceCount(n));
    return HX_OK;
}

}  // extern "C"

// ---- matrix cache --------------------------------------------------------------------------------
// A destroyed matrix keeps its streams, events, band and scratch buffers in a small parking lot; the next
// hx_create / hx_copy of the same shape on the same device takes it back after re-zeroing the state on its
// stream.  Creating and destroying a matrix costs ~0.25 ms of driver calls (3 streams, a dozen events, ~40
// stream-ordered allocations) - as much as a whole 2.5M-read ingestion chunk.  HX_NO_MATRIX_CACHE=1 disables it.
namespace {
// heap-allocated and never destroyed: a handle may be released while the process is already exiting
std::mutex &g_park_mu = *new std::mutex;
std::vector<hx_matrix *> &g_parked = *new std::vector<hx_matrix *>;
constexpr size_t HX_PARK_MAX = 4;
constexpr int64_t HX_PARK_MAX_ELEMS = (int64_t)1 << 28;      // do not sit on bands above 1 GiB
const bool g_park_on = getenv("HX_NO_MATRIX_CACHE") == nullptr;

hx_matrix *unpark(int32_t n_snps, int32_t band_w, int32_t device) {
    std::lock_guard<std::mutex> lk(g_park_mu);
    for (size_t i = 0; i < g_parked.size(); ++i) {
        hx_matrix *h = g_parked[i];
        if (h->N == n_snps && h->W == band_w && h->device == device) {
            g_parked.erase(g_parked.begin() + (long)i);
            return h;
        }
    }
    return nullptr;
}

// true if the matrix was parked (the caller must not free it)
bool park(hx_matrix *h) {
    if (!g_park_on || !h->own_stream || h->cnt_ipc || h->peer_world > 1 || h->band_elems > HX_PARK_MAX_ELEMS) return false;
    if (cudaSetDevice(h->device) != cudaSuccess) return false;
    release_counts(h);
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) return false;      // no work may outlive the handle
    hx_matrix *evict = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_park_mu);
        if (g_parked.size() >= HX_PARK_MAX) { evict = g_parked.front(); g_parked.erase(g_parked.begin()); }
        g_parked.push_back(h);
    }
    if (evict) free_all(evict);
    return true;
}

int reset_parked(hx_matrix *h) {
    HX_CUDA(cudaSetDevice(h->device));
    HX_CUDA(hx_fill_async(h->band.p, 0, sizeof(float) * (size_t)h->band_elems, h->stream));
    HX_CUDA(hx_fill_async(h->d_totals.p, 0, 8 * sizeof(unsigned long long), h->stream));
    HX_CUDA(hx_fill_async(h->d_err.p, 0, sizeof(int), h->stream));
    HX_CUDA(hx_fill_async(h->d_flags.p, 0, sizeof(hx_dev_flags), h->stream));
    h->use = {};
    return HX_OK;
}
}  // namespace

extern "C" {

int hx_create(int32_t n_snps, int32_t band_w, int32_t device, hx_matrix **out) {
    HX_CHECK_ARG(out && n_snps >= 0 && band_w >= 1);
    *out = nullptr;
    HX_CUDA(cudaSetDevice(device));
    if (hx_matrix *p = unpark(n_snps, band_w, device)) {
        const int rc = reset_parked(p);
        if (rc) { free_all(p); return rc; }
        *out = p;
        return HX_OK;
    }
    hx_matrix *h = (hx_matrix *)calloc(1, sizeof(hx_matrix));
    if (!h) return HX_E_NOMEM;
    h->N = n_snps;
    h->W = band_w;
    h->device = device;
    h->band_elems = ((int64_t)n_snps + 2) * band_w * HX_CELL;
    h->use = {};
#define HX_TRY(call)                                                                     \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess) {                                                        \
            hx_set_error("hx_create: %s -> %s", #call, cudaGetErrorString(e__));         \
            free_all(h);                                                                 \
            return e__ == cudaErrorMemoryAllocation ? HX_E_NOMEM : HX_E_CUDA;            \
        }                                                                                \
    } while (0)
    {   // keep freed blocks cached in the device's default pool (a new matrix per BAM must not pay cudaMalloc again)
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
    }
    HX_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    h->own_stream = true;
    HX_TRY(cudaEventCreate(&h->ev0));
    HX_TRY(cudaEventCreate(&h->ev1));
    HX_TRY(h->band.grow(sizeof(float) * (size_t)h->band_elems, h->stream));
    HX_TRY(hx_fill_async(h->band.p, 0, sizeof(float) * (size_t)h->band_elems, h->stream));
    HX_TRY(h->d_totals.grow(8 * sizeof(unsigned long long), h->stream));
    HX_TRY(hx_fill_async(h->d_totals.p, 0, 8 * sizeof(unsigned long long), h->stream));
    HX_TRY(h->d_err.grow(sizeof(int), h->stream));
    HX_TRY(hx_fill_async(h->d_err.p, 0, sizeof(int), h->stream));
    HX_TRY(h->scnt.grow(sizeof(double) * 8 * ((size_t)n_snps + 2), h->stream));
    HX_TRY(h->vseen.grow(sizeof(int32_t) * ((size_t)n_snps + 2), h->stream));
    HX_TRY(h->d_site.grow(sizeof(double) * 6 * ((size_t)n_snps + 2), h->stream));
    HX_TRY(h->d_flags.grow(sizeof(hx_dev_flags), h->stream));
    HX_TRY(hx_fill_async(h->d_flags.p, 0, sizeof(hx_dev_flags), h->stream));
    HX_TRY(h->d_misc.grow(32 * sizeof(double), h->stream));
    HX_TRY(h->d_run_end.grow(sizeof(int64_t) * ((size_t)n_snps + 2), h->stream));
    HX_TRY(h->d_run_list.grow(sizeof(int64_t) * (((size_t)n_snps + 3) / 2 + (size_t)n_snps + 2 + 2), h->stream));
    h->h_pinned = calloc(1, 256);     // scalars come back through pageable memory: a pinned allocation per
                                      // matrix costs more (cudaMallocHost/cudaFreeHost) than it saves
    if (!h->h_pinned) { free_all(h); return HX_E_NOMEM; }
    HX_TRY(cudaStreamSynchronize(h->stream));
#undef HX_TRY
    *out = h;
    return HX_OK;
}

int hx_destroy(hx_matrix *h) {
    if (h && !park(h)) free_all(h);
    return HX_OK;
}

int hx_copy(const hx_matrix *src, hx_matrix **out) {
    HX_CHECK_ARG(src && out);
    if (src->cnt) {
        hx_set_error("hx_copy: integer counts pending; call hx_finalize_counts first");
        return HX_E_STATE;
    }
    int rc = hx_create(src->N, src->W, src->device, out);
    if (rc) return rc;
    hx_matrix *h = *out;
    HX_CUDA(cudaStreamSynchronize(src->stream));
    HX_CUDA(cudaMemcpyAsync(h->band.p, src->band.p, sizeof(float) * (size_t)src->band_elems,
                            cudaMemcpyDeviceToDevice, h->stream));
    HX_CUDA(cudaMemcpyAsync(h->d_totals.p, src->d_totals.p, 8 * sizeof(unsigned long long),
                            cudaMemcpyDeviceToDevice, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    h->use.ingest_kernel = src->use.ingest_kernel;
    return HX_OK;
}

int hx_info(const hx_matrix *h, int32_t *n_snps, int32_t *band_w, int32_t *device) {
    HX_CHECK_ARG(h);
    if (n_snps) *n_snps = h->N;
    if (band_w) *band_w = h->W;
    if (device) *device = h->device;
    return HX_OK;
}

int hx_stream(const hx_matrix *h, void **stream) {
    HX_CHECK_ARG(h && stream);
    *stream = (void *)h->stream;
    return HX_OK;
}

int hx_set_stream(hx_matrix *h, void *stream) {
    HX_CHECK_ARG(h);
    HX_CUDA(cudaSetDevice(h->device));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    if (h->own_stream) cudaStreamDestroy(h->stream);
    h->stream = (cudaStream_t)stream;
    h->own_stream = false;
    return HX_OK;
}

int hx_sync(hx_matrix *h) {
    HX_CHECK_ARG(h);
    HX_CUDA(cudaSetDevice(h->device));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    return HX_OK;
}

// ------------------------------------------------------------------------------ ingestion
}  // extern "C"
int hx_ensure_counts_buffer(hx_matrix *h) {
    if (h->cnt) return HX_OK;
    h->cnt_elems = h->band_elems;
    HX_CUDA(cudaMallocAsync((void **)&h->cnt, sizeof(uint32_t) * (size_t)h->cnt_elems, h->stream));
    HX_CUDA(hx_fill_async(h->cnt, 0, sizeof(uint32_t) * (size_t)h->cnt_elems, h->stream));
    h->use.cnt_fresh = true;
    return HX_OK;
}
extern "C" {

int hx_set_ingest_kernel(hx_matrix *h, int which) {
    HX_CHECK_ARG(h && which >= 0 && which <= 7);
    h->use.ingest_kernel = which;
    return HX_OK;
}

int hx_set_ingest_sms(hx_matrix *h, int n_sms) {
    HX_CHECK_ARG(h && n_sms >= 0);
    h->use.ingest_sms = n_sms;
    return HX_OK;
}

int hx_ingest_device(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off,
                     const uint8_t *d_codes, int64_t n_reads) {
    HX_CHECK_ARG(h && n_reads >= 0);
    if (n_reads == 0) return HX_OK;
    HX_CHECK_ARG(d_rank && d_off && d_codes);
    HX_CUDA(cudaSetDevice(h->device));
    int rc = hx_ensure_counts_buffer(h);
    if (rc) return rc;
    return hx_launch_ingest(h, d_rank, d_off, d_codes, n_reads);
}

int hx_ingest_totals(hx_matrix *h, int64_t totals[4]) {
    HX_CHECK_ARG(h && totals);
    HX_CUDA(cudaSetDevice(h->device));
    unsigned long long *hp = (unsigned long long *)h->h_pinned;
    int *he = (int *)(hp + 8);
    HX_CUDA(cudaMemcpyAsync(hp, h->d_totals.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaMemcpyAsync(he, h->d_err.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (h->use.prepass_ran) HX_CUDA(cudaMemcpyAsync(he + 1, &h->d_flags.p->ingest_sorted, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    if (h->use.prepass_ran && he[1] == 0) hx_note_unsorted();
    hx_wire_trace_dump();
    if (h->use.ev_rec) cudaEventElapsedTime(&h->use.last_ms[0], h->ev0, h->ev1);
    for (int i = 0; i < 4; ++i) totals[i] = (int64_t)hp[i];
    if (*he) {
        hx_set_error("ingest: invalid packed read(s): %s%s",
                     (*he & 1) ? "[read leaves [0,N] or has more SNPs than band_w+1] " : "",
                     (*he & 2) ? "[allele code > 6]" : "");
        return HX_E_READ;
    }
    return HX_OK;
}

int hx_ingest_host(hx_matrix *h, const int32_t *rank, const int64_t *off, const uint8_t *codes,
                   int64_t n_reads, int64_t totals[4]) {
    HX_CHECK_ARG(h && totals && n_reads >= 0);
    HX_CUDA(cudaSetDevice(h->device));
    // Large inputs travel in chunks so that the copy of chunk i+1 overlaps the expansion of chunk i.  Default
    // ("slim"): the allele bytes are copied as they are, straight from the caller's memory, while a few host threads
    // turn the chunk's int32 ranks and int64 offsets (12 of the 27 bytes per read of a 150 bp metagenome) into uint8
    // rank deltas and SNP counts (2 bytes per read); the device rebuilds rank / offsets with one scan.
    // HX_HOST_PIPELINE=dense: the alleles are re-encoded too (2 bits each) - fewer bytes, but one pass over every
    // allele on the host (measured on the 16-core GPU box: 11.9 ms per 10M reads against 5.3 ms as they are);
    // HX_HOST_PIPELINE=packed: the three arrays as they are in 4 chunks; =off: one copy, one launch.
    const char *pipe_env = getenv("HX_HOST_PIPELINE");
    const bool want_dense = pipe_env && !strcmp(pipe_env, "dense");
    const bool want_slim = !pipe_env || !strcmp(pipe_env, "slim");       // default
    if (n_reads >= 200000 && rank && off && codes && (want_dense || want_slim)) {
        int64_t done = 0;
        const int rc = hx_ingest_host_pipelined(h, rank, off, codes, n_reads, !want_dense, &done);
        if (rc == HX_OK) return hx_ingest_totals(h, totals);
        if (rc != HX_E_STATE) return rc;            // HX_E_STATE: not sorted by rank from read `done` on -> the rest of
        hx_note_unsorted();
        rank += done; off += done; n_reads -= done; //               the packed arrays as they are (counts just add up)
    }
    if (n_reads > 0) {
        HX_CHECK_ARG(rank && off && codes);
        const int64_t n_codes = off[n_reads] - off[0];
        HX_CHECK_ARG(n_codes >= 0);
        HX_CUDA(h->s_rank.grow(sizeof(int32_t) * n_reads, h->stream));
        HX_CUDA(h->s_off.grow(sizeof(int64_t) * (n_reads + 1) + 16, h->stream));
        HX_CUDA(h->s_codes.grow(n_codes + 16, h->stream));
        int rc = hx_ensure_counts_buffer(h);
        if (rc) return rc;
        const int n_chunks = n_reads >= 200000 && !(pipe_env && !strcmp(pipe_env, "off")) ? 4 : 1;
        if (n_chunks > 1 && !h->copy_stream) HX_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        cudaStream_t cs = n_chunks > 1 ? h->copy_stream : h->stream;
        if (n_chunks > 1) {
            // the staging buffers may have just been (re)allocated on the compute stream
            if (!h->host_ev) HX_CUDA(cudaEventCreateWithFlags(&h->host_ev, cudaEventDisableTiming));
            HX_CUDA(cudaEventRecord(h->host_ev, h->stream));
            HX_CUDA(cudaStreamWaitEvent(cs, h->host_ev, 0));
        }
        int64_t a = 0;
        for (int c = 0; c < n_chunks; ++c) {
            const int64_t b = hx_chunk_end(off, a, n_reads, n_codes, c, n_chunks);
            if (b <= a && c + 1 < n_chunks) continue;
            HX_CUDA(cudaMemcpyAsync(h->s_rank.p + a, rank + a, sizeof(int32_t) * (size_t)(b - a), cudaMemcpyHostToDevice, cs));
            HX_CUDA(cudaMemcpyAsync(h->s_off.p + a, off + a, sizeof(int64_t) * (size_t)(b - a + 1), cudaMemcpyHostToDevice, cs));
            HX_CUDA(cudaMemcpyAsync(h->s_codes.p + (off[a] - off[0]), codes + off[a], (size_t)(off[b] - off[a]), cudaMemcpyHostToDevice, cs));
            if (n_chunks > 1) {
                HX_CUDA(cudaEventRecord(h->host_ev, cs));
                HX_CUDA(cudaStreamWaitEvent(h->stream, h->host_ev, 0));
            }
            // kernels index codes by absolute offsets: bias the base pointer by off[0]
            rc = hx_launch_ingest(h, h->s_rank.p + a, h->s_off.p + a, h->s_codes.p - off[0], b - a);
            if (rc) return rc;
            a = b;
        }
    }
    return hx_ingest_totals(h, totals);
}

int hx_ingest_host_compact(hx_matrix *h, const int32_t *rank, const uint16_t *klen, const uint8_t *codes4,
                           int64_t n_reads, int64_t n_codes, int64_t totals[4]) {
    HX_CHECK_ARG(h && totals && n_reads >= 0 && n_codes >= 0);
    HX_CUDA(cudaSetDevice(h->device));
    if (n_reads > 0) {
        HX_CHECK_ARG(rank && klen && (codes4 || n_codes == 0));
        cudaStream_t st = h->stream;
        const int64_t n_words = (n_codes + 7) / 8;          // 32-bit words of packed nibbles
        constexpr int ITEMS = 16;
        const int64_t n1 = n_reads + 1;
        const int64_t nblk = (n1 + 256 * ITEMS - 1) / (256 * ITEMS);
        HX_CUDA(h->s_rank.grow(sizeof(int32_t) * n_reads, st));
        HX_CUDA(h->s_off.grow(sizeof(int64_t) * n1 + 16, st));
        HX_CUDA(h->s_codes.grow(n_words * 8 + 16, st));
        HX_CUDA(h->s_klen.grow(sizeof(uint16_t) * n_reads, st));
        HX_CUDA(h->s_codes4.grow(sizeof(uint32_t) * n_words, st));
        HX_CUDA(h->s_scan.grow(sizeof(int64_t) * nblk, st));
        HX_CUDA(cudaMemcpyAsync(h->s_rank.p, rank, sizeof(int32_t) * (size_t)n_reads, cudaMemcpyHostToDevice, st));
        HX_CUDA(cudaMemcpyAsync(h->s_klen.p, klen, sizeof(uint16_t) * (size_t)n_reads, cudaMemcpyHostToDevice, st));
        if (n_codes)
            HX_CUDA(cudaMemcpyAsync(h->s_codes4.p, codes4, (size_t)((n_codes + 1) / 2), cudaMemcpyHostToDevice, st));
        // off = exclusive scan of klen (n+1 entries, off[n] = n_codes); codes = one byte per nibble
        k_widen_klen<<<(unsigned)((n1 + 255) / 256), 256, 0, st>>>(h->s_klen.p, n_reads, h->s_off.p);
        k_scan_partials<int64_t, 0, ITEMS><<<(unsigned)nblk, 256, 0, st>>>(h->s_off.p, n1, h->s_scan.p);
        k_scan_spine<int64_t, 0><<<1, 32, 0, st>>>(h->s_scan.p, nblk, nullptr);
        k_scan_apply<int64_t, 0, ITEMS, true><<<(unsigned)nblk, 256, 0, st>>>(h->s_off.p, n1, h->s_scan.p, h->s_off.p);
        if (n_words)
            k_unpack_nibbles<<<(unsigned)((n_words + 255) / 256), 256, 0, st>>>(h->s_codes4.p, n_words, (uint2 *)h->s_codes.p);
        h->use.launches += 5;
        HX_CUDA(cudaGetLastError());
        int rc = hx_ensure_counts_buffer(h);
        if (rc) return rc;
        rc = hx_launch_ingest(h, h->s_rank.p, h->s_off.p, h->s_codes.p, n_reads);
        if (rc) return rc;
    }
    return hx_ingest_totals(h, totals);
}

int hx_counts_buffer(hx_matrix *h, void **d_counts, int64_t *n_u32, void **d_totals, int64_t *n_i64) {
    HX_CHECK_ARG(h && d_counts && n_u32 && d_totals && n_i64);
    HX_CUDA(cudaSetDevice(h->device));
    int rc = hx_ensure_counts_buffer(h);
    if (rc) return rc;
    *d_counts = h->cnt;
    h->use.cnt_fresh = false;             // the caller may write through the pointer (until the next hx_reset_counts)
    *n_u32 = h->cnt_elems;
    *d_totals = h->d_totals.p;
    *n_i64 = 4;
    return HX_OK;
}

int hx_counts_pack(hx_matrix *h, int32_t world, void **d_packed, int64_t *n_u32) {
    HX_CHECK_ARG(h && d_packed && n_u32 && world >= 1 && world <= 65535);
    HX_CUDA(cudaSetDevice(h->device));
    int rc = hx_ensure_counts_buffer(h);
    if (rc) return rc;
    const int64_t n_pairs = h->band_elems / HX_CELL;
    const int64_t flag_at = (n_pairs * HX_PACK_WORDS + 3) & ~(int64_t)3;      // 16-byte aligned trailer
    const int64_t words = flag_at + 4;
    HX_CUDA(h->d_pack.grow(sizeof(uint32_t) * words, h->stream));
    HX_CUDA(hx_fill_async(h->d_pack.p + n_pairs * HX_PACK_WORDS, 0, (size_t)(words - n_pairs * HX_PACK_WORDS) * 4, h->stream));
    const int64_t n_w = n_pairs * HX_PACK_WORDS;
    k_pack_counts<<<(unsigned)((n_w + 255) / 256), 256, 0, h->stream>>>(h->cnt, n_pairs, 65535u / (uint32_t)world,
                                                                        h->d_pack.p, flag_at);
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    *d_packed = h->d_pack.p;
    *n_u32 = words;
    return HX_OK;
}

int hx_counts_unpack(hx_matrix *h, int32_t *overflowed) {
    HX_CHECK_ARG(h && overflowed && h->d_pack.p && h->cnt);
    HX_CUDA(cudaSetDevice(h->device));
    const int64_t n_pairs = h->band_elems / HX_CELL;
    const int64_t flag_at = (n_pairs * HX_PACK_WORDS + 3) & ~(int64_t)3;
    const int64_t n_w = n_pairs * HX_PACK_WORDS;
    h->use.cnt_fresh = false;
    k_unpack_counts<<<(unsigned)((n_w + 255) / 256), 256, 0, h->stream>>>(h->d_pack.p, n_pairs, h->cnt, flag_at);
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    uint32_t *hp = (uint32_t *)h->h_pinned + 40;
    HX_CUDA(cudaMemcpyAsync(hp, h->d_pack.p + flag_at, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    *overflowed = *hp != 0;
    return HX_OK;
}

int hx_counts_unpack_async(hx_matrix *h, void *stream) {
    HX_CHECK_ARG(h && h->d_pack.p && h->cnt);
    HX_CUDA(cudaSetDevice(h->device));
    const int64_t n_pairs = h->band_elems / HX_CELL;
    const int64_t flag_at = (n_pairs * HX_PACK_WORDS + 3) & ~(int64_t)3;
    const int64_t n_w = n_pairs * HX_PACK_WORDS;
    h->use.cnt_fresh = false;
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    k_unpack_counts<<<(unsigned)((n_w + 255) / 256), 256, 0, st>>>(h->d_pack.p, n_pairs, h->cnt, flag_at);
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    return HX_OK;
}

int hx_counts_pack_overflowed(hx_matrix *h, int32_t *overflowed) {
    HX_CHECK_ARG(h && overflowed && h->d_pack.p);
    HX_CUDA(cudaSetDevice(h->device));
    const int64_t n_pairs = h->band_elems / HX_CELL;
    const int64_t flag_at = (n_pairs * HX_PACK_WORDS + 3) & ~(int64_t)3;
    uint32_t *hp = (uint32_t *)h->h_pinned + 40;
    HX_CUDA(cudaMemcpyAsync(hp, h->d_pack.p + flag_at, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    *overflowed = *hp != 0;
    return HX_OK;
}

__global__ void k_counts_max(const uint32_t *__restrict__ cnt, int64_t n, uint32_t *__restrict__ out) {
    uint32_t m = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = max(m, cnt[i]);
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

int hx_counts_max(hx_matrix *h, uint32_t *max_count) {
    HX_CHECK_ARG(h && max_count);
    HX_CUDA(cudaSetDevice(h->device));
    int rc = hx_ensure_counts_buffer(h);
    if (rc) return rc;
    uint32_t *d_out = &h->d_flags.p->counts_max;
    HX_CUDA(hx_fill_async(d_out, 0, sizeof(uint32_t), h->stream));
    k_counts_max<<<592, 256, 0, h->stream>>>(h->cnt, h->cnt_elems, d_out);
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    uint32_t *hp = (uint32_t *)h->h_pinned + 41;
    HX_CUDA(cudaMemcpyAsync(hp, d_out, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    *max_count = *hp;
    return HX_OK;
}

int hx_counts_ipc_export(hx_matrix *h, int32_t world, void *handle_out) {
    HX_CHECK_ARG(h && handle_out && world >= 1 && world <= HX_MAX_PEERS);
    HX_CUDA(cudaSetDevice(h->device));
    release_counts(h);
    const int64_t rows = (int64_t)h->N + 2;
    const int64_t rows_per = (rows + world - 1) / world;
    h->cnt_elems = rows_per * world * h->W * HX_CELL;          // padded so that every rank owns rows_per rows
    HX_CUDA(cudaMalloc((void **)&h->cnt, sizeof(uint32_t) * (size_t)h->cnt_elems));   // IPC needs a plain allocation
    h->cnt_ipc = true;
    h->use.cnt_fresh = false;
    HX_CUDA(hx_fill_async(h->cnt, 0, sizeof(uint32_t) * (size_t)h->cnt_elems, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    cudaIpcMemHandle_t hd;
    HX_CUDA(cudaIpcGetMemHandle(&hd, h->cnt));
    memcpy(handle_out, &hd, sizeof(hd));
    h->peer_rows_per = (int)rows_per;
    return HX_OK;
}

int hx_counts_ipc_import(hx_matrix *h, const void *handles, int32_t world, int32_t my_rank) {
    HX_CHECK_ARG(h && handles && world >= 1 && world <= HX_MAX_PEERS && my_rank >= 0 && my_rank < world);
    if (!h->cnt_ipc) { hx_set_error("hx_counts_ipc_import: call hx_counts_ipc_export first"); return HX_E_STATE; }
    HX_CUDA(cudaSetDevice(h->device));
    for (int g = 0; g < world; ++g) {
        if (g == my_rank) { h->peer_host[g] = h->cnt; continue; }
        cudaIpcMemHandle_t hd;
        memcpy(&hd, (const char *)handles + (size_t)g * sizeof(hd), sizeof(hd));
        void *p = nullptr;
        HX_CUDA(cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
        h->ipc_opened[g] = p;
        h->peer_host[g] = (uint32_t *)p;
    }
    if (!h->d_peer_tbl) HX_CUDA(cudaMalloc((void **)&h->d_peer_tbl, sizeof(uint32_t *) * HX_MAX_PEERS));
    HX_CUDA(cudaMemcpy(h->d_peer_tbl, h->peer_host, sizeof(uint32_t *) * HX_MAX_PEERS, cudaMemcpyHostToDevice));
    h->peer_world = world;
    return HX_OK;
}

int hx_counts_ipc_close(hx_matrix *h) {
    HX_CHECK_ARG(h);
    HX_CUDA(cudaSetDevice(h->device));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    for (int g = 0; g < HX_MAX_PEERS; ++g) {
        if (h->ipc_opened[g]) HX_CUDA(cudaIpcCloseMemHandle(h->ipc_opened[g]));
        h->ipc_opened[g] = nullptr;
        h->peer_host[g] = nullptr;
    }
    h->peer_world = 0;                          // counts go to the local buffer again
    return HX_OK;
}

int hx_reset_counts(hx_matrix *h) {
    HX_CHECK_ARG(h);
    HX_CUDA(cudaSetDevice(h->device));
    // one launch: the counts, the eight totals and the error word
    if (h->cnt) {
        const size_t n16 = (sizeof(uint32_t) * (size_t)h->cnt_elems + 15) / 16;
        const size_t want = (n16 + 255) / 256;
        const unsigned grid = (unsigned)(want < 1 ? 1 : (want > 148 * 16 ? 148 * 16 : want));
        k_reset_counts<<<grid, 256, 0, h->stream>>>(reinterpret_cast<uint4 *>(h->cnt), sizeof(uint32_t) * (size_t)h->cnt_elems,
                                                    h->d_totals.p, h->d_err.p);
        HX_CUDA(cudaGetLastError());
        h->use.cnt_fresh = true;
    } else {
        HX_CUDA(hx_fill_async(h->d_totals.p, 0, 8 * sizeof(unsigned long long), h->stream));
        HX_CUDA(hx_fill_async(h->d_err.p, 0, sizeof(int), h->stream));
    }
    return HX_OK;
}

int hx_finalize_counts(hx_matrix *h) {
    HX_CHECK_ARG(h);
    if (!h->cnt) return HX_OK;
    HX_CUDA(cudaSetDevice(h->device));
    const int64_t n = h->band_elems;
    k_fold_counts<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->cnt, h->band.p, n);
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    if (h->cnt_ipc) HX_CUDA(cudaStreamSynchronize(h->stream));   // a shared allocation is freed with cudaFree
    release_counts(h);                                           // (stream-ordered otherwise: no host wait here)
    h->use.counts_dirty = true;
    return HX_OK;
}

// ------------------------------------------------------------------------------ scalar surface
int hx_add_observation(hx_matrix *h, int a, int b, int32_t i, int32_t j, float amount) {
    HX_CHECK_ARG(h);
    int rc = in_band(h, a, b, i, j);
    if (rc) { hx_set_error("add_observation(%d,%d,%d,%d): outside band/arguments", a, b, i, j); return rc; }
    HX_CUDA(cudaSetDevice(h->device));
    k_add_one<<<1, 1, 0, h->stream>>>(h->band.p + hx_cell_off(h->W, i, j) + a * HX_NSYM + b, amount);
    h->use.launches++;
    h->use.counts_dirty = true;
    HX_CUDA(cudaGetLastError());
    return HX_OK;
}

int hx_get_observation(hx_matrix *h, int a, int b, int32_t i, int32_t j, float *out) {
    HX_CHECK_ARG(h && out);
    int rc = in_band(h, a, b, i, j);
    if (rc == HX_E_BAND) { *out = 0.0f; return HX_E_BAND; }
    if (rc) { hx_set_error("get_observation(%d,%d,%d,%d): bad arguments", a, b, i, j); return rc; }
    HX_CUDA(cudaSetDevice(h->device));
    const int64_t o = hx_cell_off(h->W, i, j) + a * HX_NSYM + b;
    float v = 0.0f;
    HX_CUDA(cudaMemcpyAsync(&v, h->band.p + o, sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    if (h->cnt) {       // counts not folded yet: report the sum
        uint32_t c = 0;
        HX_CUDA(cudaMemcpyAsync(&c, h->cnt + o, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
        HX_CUDA(cudaStreamSynchronize(h->stream));
        v += (float)c;
    }
    *out = v;
    return HX_OK;
}

int hx_reweight_observation(hx_matrix *h, int a, int b, int32_t i, int32_t j, double ratio,
                            double *removed) {
    HX_CHECK_ARG(h && removed);
    int rc = in_band(h, a, b, i, j);
    if (rc == HX_E_BAND) { *removed = 0.0; return HX_E_BAND; }
    if (rc) { hx_set_error("reweight_observation(%d,%d,%d,%d): bad arguments", a, b, i, j); return rc; }
    if (h->cnt) { hx_set_error("reweight_observation: call hx_finalize_counts first"); return HX_E_STATE; }
    HX_CUDA(cudaSetDevice(h->device));
    k_reweight_one<<<1, 1, 0, h->stream>>>(h->band.p + hx_cell_off(h->W, i, j) + a * HX_NSYM + b, ratio, h->d_misc.p + 16);
    h->use.launches++;
    h->use.counts_dirty = true;
    HX_CUDA(cudaGetLastError());
    HX_CUDA(cudaMemcpyAsync(removed, h->d_misc.p + 16, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    return HX_OK;
}

// ------------------------------------------------------------------------------ bulk I/O
int hx_band_to_host(hx_matrix *h, float *out) {
    HX_CHECK_ARG(h && out);
    if (h->cnt) { hx_set_error("band_to_host: call hx_finalize_counts first"); return HX_E_STATE; }
    HX_CUDA(cudaSetDevice(h->device));
    HX_CUDA(cudaMemcpyAsync(out, h->band.p, sizeof(float) * (size_t)h->band_elems, cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    return HX_OK;
}

int hx_band_from_host(hx_matrix *h, const float *in) {
    HX_CHECK_ARG(h && in);
    if (h->cnt) { hx_set_error("band_from_host: call hx_finalize_counts first"); return HX_E_STATE; }
    HX_CUDA(cudaSetDevice(h->device));
    HX_CUDA(cudaMemcpyAsync(h->band.p, in, sizeof(float) * (size_t)h->band_elems, cudaMemcpyHostToDevice, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    h->use.counts_dirty = true;
    return HX_OK;
}

int hx_to_dense(hx_matrix *h, float *out) {
    HX_CHECK_ARG(h && out);
    const int64_t P = (int64_t)h->N + 2;
    float *tmp = (float *)malloc(sizeof(float) * (size_t)h->band_elems);
    if (!tmp) return HX_E_NOMEM;
    int rc = hx_band_to_host(h, tmp);
    if (rc) { free(tmp); return rc; }
    memset(out, 0, sizeof(float) * (size_t)(HX_CELL * P * P));
    for (int64_t pj = 1; pj < P; ++pj)
        for (int64_t d = 1; d <= h->W && pj - d >= 0; ++d) {
            const float *cell = tmp + hx_cell_off(h->W, pj - d, pj);
            for (int ab = 0; ab < HX_CELL; ++ab) out[(ab * P + (pj - d)) * P + pj] = cell[ab];
        }
    free(tmp);
    return HX_OK;
}

int hx_last_kernel_ms(hx_matrix *h, int which, float *ms) {
    HX_CHECK_ARG(h && ms && which >= 0 && which < 5);
    *ms = h->use.last_ms[which];
    return HX_OK;
}

int hx_launch_count(const hx_matrix *h, int64_t *n) {
    HX_CHECK_ARG(h && n);
    *n = h->use.launches;
    return HX_OK;
}

}  // extern "C"
