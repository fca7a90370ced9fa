// Internal definitions shared by the translation units of libhanselx.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <algorithm>

#include "hanselx.h"

#define HX_NSYM 7
#define HX_CELL 49
#define HX_SYM_N 4
#define HX_SYM_DEL 5
#define HX_SYM_GAP 6   // '_'
#define HX_RING 4096   // lookback window of chosen symbols kept in shared memory by the walk
#define HX_MAX_L (HX_RING - 1)

#define HX_MAX_PEERS 8
// Where count increments go: the local partial band, or - with the fused multi-GPU exchange - the GPU
// that owns band row pj (rows are dealt out in contiguous blocks of rows_per), reached through NVLink
// peer memory.  Passed to the ingestion kernels by value.
struct HxCnt {
    uint32_t *local;
    uint32_t *const *peer;           // device array [world] of every rank's buffer (own entry included)
    int world, rows_per;
#ifdef __CUDACC__
    __device__ __forceinline__ uint32_t *cell(int64_t W, int64_t pi, int64_t pj) const {
        uint32_t *base = local;
        if (world > 1) base = peer[pj / rows_per];
        return base + (pj * W + (pj - pi - 1)) * 49;
    }
    // The target as a kernel instantiation sees it: FUSED = false (a single-GPU build) folds the peer path away.
    template <bool FUSED>
    __device__ __forceinline__ HxCnt for_build() const {
        HxCnt c = *this;
        if (!FUSED) { c.world = 1; c.rows_per = 1; c.peer = nullptr; }
        return c;
    }
#endif
};

// A stream-ordered device buffer of T that grows on demand; all zero is empty (hx_matrix is calloc'ed).  cap is the
// size of the allocation in bytes.  grow() allocates exactly the bytes asked for: a caller that wants headroom adds it.
template <class T>
struct HxDevBuf {
    T *p;
    int64_t cap;
    // bytes > cap: free the old block (its contents are not kept) and allocate `bytes` on st; *grew is set if so
    cudaError_t grow(int64_t bytes, cudaStream_t st, bool *grew = nullptr) {
        if (bytes <= cap) return cudaSuccess;
        if (grew) *grew = true;
        release(st);
        const cudaError_t e = cudaMallocAsync((void **)&p, (size_t)bytes, st);
        if (e != cudaSuccess) { p = nullptr; return e; }
        cap = bytes;
        return cudaSuccess;
    }
    void release(cudaStream_t st) {
        if (p) cudaFreeAsync(p, st);
        p = nullptr;
        cap = 0;
    }
};

// The device flag word of a matrix (hx_matrix::d_flags), shared by recovery and ingestion.
struct hx_dev_flags {
    int hole_site;                   // recovery: the site without a candidate (0 once a walk reached site N)
    int hole;                        // recovery: a walk met a hole; every later recovery kernel of the launch is a no-op
    int q_unsafe;                    // recovery: a walk term does not fit the fixed-point tables
    int walk_redone;                 // sites the parallel-in-time walk walked again since hx_create (hx_debug_walk_redone)
    int ingest_sorted;               // ingestion: the pre-pass verdict, non-zero = reads sorted by rank
    int fallback_go;                 // ingestion: non-zero = the counting-sort fallback runs
    uint32_t counts_max;             // hx_counts_max
    int score_err;                   // path scoring: a haplotype code > 6 at a site, or not '_' at site 0
};
static_assert(sizeof(hx_dev_flags) == 8 * sizeof(int), "hx_dev_flags is one int[8]");

// What recovery reports for one haplotype (hx_matrix::d_stats).
struct hx_hap_stats {
    double hp_current, hp_original;  // ordered log10 sums of the path's marginals in the current / original matrix
    double min_marginal, ratio, removed;
    double done;                     // 1.0: the walk reached site N and the statistics are complete
    double pad[2];
};
static_assert(sizeof(hx_hap_stats) == 64, "hx_hap_stats is one double[8]");

#define HX_WIRE_SETS 3
// One staging set of the dense wire format (wire.cu): raw shipped bytes + the rebuilt packed arrays
struct hx_wire_set {
    HxDevBuf<uint8_t> raw; HxDevBuf<int32_t> rank; HxDevBuf<int64_t> off; HxDevBuf<uint8_t> codes;
    HxDevBuf<int64_t> partials, run_end;
    cudaEvent_t copied, decoded, consumed;
};

struct hx_matrix {
    int32_t N, W, device;
    int64_t band_elems;              // (N+2)*W*49
    cudaStream_t stream;
    bool own_stream;
    HxDevBuf<float> band;            // float32 working matrix (what the Hansel surface reads)
    uint32_t *cnt;                   // integer counts being ingested (lazily allocated)
    bool cnt_ipc;                    // cnt is a plain cudaMalloc allocation shared through CUDA IPC
    int64_t cnt_elems;               // allocated uint32 elements (>= band_elems; padded for the fused exchange)
    uint32_t *peer_host[HX_MAX_PEERS];   // fused exchange: every rank's cnt (own entry = local pointer)
    uint32_t **d_peer_tbl;           // the same table on the device
    int peer_world, peer_rows_per;
    void *ipc_opened[HX_MAX_PEERS];  // pointers returned by cudaIpcOpenMemHandle (to close)
    HxDevBuf<unsigned long long> d_totals;   // [8] slices, crumbs, covered, sentinels, -, -, -, -
    HxDevBuf<int> d_err;             // ingestion error bits
    // staging for hx_ingest_host
    HxDevBuf<int32_t> s_rank; HxDevBuf<int64_t> s_off; HxDevBuf<uint8_t> s_codes;
    HxDevBuf<uint16_t> s_klen; HxDevBuf<uint32_t> s_codes4; HxDevBuf<int64_t> s_scan;   // compact wire format staging
    hx_wire_set wire[HX_WIRE_SETS];  // dense wire format: rotating staging sets
    cudaStream_t copy_stream, decode_stream; // host->device copies / decode kernels of the dense format
    uint8_t *pin[2]; int64_t pin_cap[2]; cudaEvent_t pin_ev[2]; bool pin_busy[2];   // pinned encode buffers of hx_ingest_host
    // recovery scratch
    HxDevBuf<double> scnt;           // (N+2)*8 per-site counts + total
    HxDevBuf<int32_t> vseen;         // (N+2) valid symbols seen per site
    HxDevBuf<uint8_t> d_path;        // path buffer(s)
    HxDevBuf<hx_hap_stats> d_stats;  // per-haplotype stats
    HxDevBuf<double> d_site;         // 2 x 3*(N+2) per-site log10 marginal (cur), (orig), marginal (alternating haplotypes)
    cudaStream_t sum_stream;         // the ordered log10 sums of a haplotype run here, off the critical path
    cudaEvent_t sum_done[2], site_ready;
    // walk tables (recover.cu): (N+2)*Lw*56 log10 lookback terms, (N+2)*8 log10 marginals, and their int32
    // fixed-point twins for the quantised walk
    HxDevBuf<double> terms, logm;
    HxDevBuf<int32_t> termsq, logmq;
    // parallel-in-time walk: speculative block paths, the majority-allele guess, per-start results and start picks
    HxDevBuf<uint8_t> spec, guess;
    HxDevBuf<int> spec_ok, cand_idx;
    HxDevBuf<double> d_partials;     // block partials of the reweight reduction
    HxDevBuf<hx_dev_flags> d_flags;
    HxDevBuf<int64_t> d_run_end;     // (N+1) end (exclusive) of the run of reads with each rank
    HxDevBuf<int64_t> d_run_list;    // compact run list for the tensor-core kernel: ranks (int32), stops (int64), count
    HxDevBuf<int4> d_jobs;           // per-CTA job tables of the tensor-core kernel (ingest_umma.cu)
    HxDevBuf<double> d_misc;         // small outputs (weights etc.)
    HxDevBuf<uint32_t> d_pack;       // packed counts for the cross-GPU exchange (api.cu)
    // read support (support.cu): haplotype codes and bit-planes, the sums, one chunk of reads, per-read results
    HxDevBuf<uint8_t> a_haps; HxDevBuf<uint4> a_planes; HxDevBuf<unsigned long long> a_sums;
    HxDevBuf<int32_t> a_rank; HxDevBuf<int64_t> a_off; HxDevBuf<uint8_t> a_codes; HxDevBuf<int32_t> a_best;
    cudaEvent_t a_ev[2];             // times the assignment kernels (hx_last_kernel_ms which = 3)
    // path scoring (score.cu): haplotype codes, per-site outputs of one chunk of haplotypes, per-haplotype sums
    HxDevBuf<uint8_t> sc_haps, sc_best; HxDevBuf<double> sc_site, sc_ll; HxDevBuf<int32_t> sc_cnt;
    cudaEvent_t sc_ev[2];            // times the scoring kernels (hx_last_kernel_ms which = 4)
    void *h_pinned;                  // small host buffer for D2H of scalars
    void *lr_scratch;                // long-read ingestion scratch (ingest_long.cu)
    void *l2_scratch;                // long-read tensor-core ingestion scratch (ingest_lumma.cu)
    cudaEvent_t ev0, ev1;
    cudaEvent_t host_ev;             // orders the chunked host->device copies of hx_ingest_host
    // State of one use of the handle.  A new matrix and a parked one taken back by hx_create both start from `use = {}`.
    struct Use {
        int64_t launches = 0;
        int ingest_kernel = 0;
        int ingest_sms = 0;          // SMs the persistent ingestion kernels may use (0 = all)
        bool counts_dirty = true;    // scnt / vseen do not reflect the band yet
        bool cnt_fresh = false;      // cnt is still all zero (nothing ingested / received since it was cleared)
        bool ev_rec = false;         // ev0/ev1 have been recorded at least once
        bool prepass_ran = false;    // d_flags->ingest_sorted holds the sortedness verdict of the last ingestion launch
        int wire_next = 0;           // the next staging set of the dense wire format
        bool sum_busy[2] = {};       // sum_done[b] marks ordered sums not yet joined into the main stream
        float last_ms[5] = {};
    } use;
};

void hx_set_error(const char *fmt, ...);

#define HX_CUDA(call)                                                                   \
    do {                                                                                \
        cudaError_t e__ = (call);                                                       \
        if (e__ != cudaSuccess) {                                                       \
            hx_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return HX_E_CUDA;                                                           \
        }                                                                               \
    } while (0)

#define HX_CHECK_ARG(cond)                                                              \
    do {                                                                                \
        if (!(cond)) {                                                                  \
            hx_set_error("%s:%d argument check failed: %s", __FILE__, __LINE__, #cond); \
            return HX_E_ARG;                                                            \
        }                                                                               \
    } while (0)

// Fills run as kernels, not cudaMemsetAsync: a memset may be queued on a copy engine behind the multi-megabyte
// host->device copies of the overlapped ingestion (measured: +0.08 ms per ingestion launch while a copy is in flight).
#ifdef __CUDACC__
static __global__ void k_fill_bytes(uint8_t *p, unsigned v, size_t bytes) {
    if (reinterpret_cast<uintptr_t>(p) & 15) {        // unaligned (small) fills: plain byte stores
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < bytes; i += (size_t)gridDim.x * blockDim.x)
            p[i] = (uint8_t)v;
        return;
    }
    const size_t n16 = bytes / 16;
    const uint4 w = make_uint4(v, v, v, v);
    uint4 *p16 = reinterpret_cast<uint4 *>(p);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) p16[i] = w;
    if (blockIdx.x == 0)
        for (size_t i = n16 * 16 + threadIdx.x; i < bytes; i += blockDim.x) p[i] = (uint8_t)v;
}
static inline cudaError_t hx_fill_async(void *p, int byte, size_t bytes, cudaStream_t st) {
    if (!bytes) return cudaSuccess;
    const unsigned b = (unsigned)byte & 0xffu, v = b * 0x01010101u;
    const size_t want = (bytes / 16 + 255) / 256;
    const unsigned grid = (unsigned)(want < 1 ? 1 : (want > 148 * 16 ? 148 * 16 : want));
    k_fill_bytes<<<grid, 256, 0, st>>>(static_cast<uint8_t *>(p), v, bytes);
    return cudaGetLastError();
}
#endif

__host__ __device__ __forceinline__ int64_t hx_cell_off(int64_t W, int64_t pi, int64_t pj) {
    return (pj * W + (pj - pi - 1)) * HX_CELL;
}

// Host arrays sent in n_chunks chunks of about equal code counts, cut at read boundaries: the end (exclusive) of
// chunk c, which starts at read a.  The last chunk ends at n_reads; an earlier one may come out empty (end <= a).
static inline int64_t hx_chunk_end(const int64_t *off, int64_t a, int64_t n_reads, int64_t n_codes, int c, int n_chunks) {
    if (c + 1 == n_chunks) return n_reads;
    return std::lower_bound(off + a, off + n_reads, off[0] + n_codes * (c + 1) / n_chunks) - off;
}

#ifdef __CUDACC__
// mbarriers and 1-D TMA bulk copies into this CTA's shared memory (addresses are shared-window addresses)
__device__ __forceinline__ uint32_t hx_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void hx_mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void hx_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void hx_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "HX_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra HX_DONE_%=;\n\t"
        "bra HX_WAIT_%=;\n\t"
        "HX_DONE_%=:\n\t}" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// src must be 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void hx_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
#endif

// ingest.cu
int hx_launch_ingest(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off,
                     const uint8_t *d_codes, int64_t n_reads);
int hx_launch_ingest_presorted(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off,
                               const uint8_t *d_codes, int64_t n_reads, int64_t *run_end, const int *ok);
// ingest_umma.cu
bool hx_umma_possible(const hx_matrix *h);
int hx_launch_ingest_umma(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off, const uint8_t *d_codes,
                          int64_t n_reads, const int64_t *run_end, const int *sorted_flag);
// api.cu
HxCnt hx_cnt_ref(const hx_matrix *h);
int hx_ensure_counts_buffer(hx_matrix *h);
// wire.cu
void hx_wire_free(hx_matrix *h);
void hx_wire_trace_dump();
// set once an ingestion of this process met reads that were not sorted by rank (hx_ingest_totals reads the pre-pass
// verdict back; hx_ingest_host knows from its own pass): later short-read launches queue the counting-sort tensor-core
// kernel (ingest_lumma.cu) as their unsorted-input fallback instead of one RED per pair
bool hx_unsorted_seen();
void hx_note_unsorted();
int hx_ingest_host_pipelined(hx_matrix *h, const int32_t *rank, const int64_t *off, const uint8_t *codes, int64_t n_reads,
                             bool slim, int64_t *done_reads);
// ingest_long.cu
int hx_launch_ingest_long(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off,
                          const uint8_t *d_codes, int64_t n_reads, const int *sorted_flag);
void hx_lr_free(hx_matrix *h);
// ingest_lumma.cu
int hx_launch_ingest_lumma(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off, const uint8_t *d_codes,
                           int64_t n_reads, const int *go);
int64_t hx_lumma_scratch_bytes(const hx_matrix *h, int64_t n_reads);
void hx_l2_free(hx_matrix *h);
// recover.cu
int hx_ensure_counts(hx_matrix *h);
// support.cu
void hx_support_free(hx_matrix *h);
// score.cu
void hx_score_free(hx_matrix *h);
