// Helpers shared by the ingestion kernels (ingest.cu, ingest_umma.cu, ingest_lumma.cu, ingest_long.cu): the per-read
// rules of the reference (which reads count, the sentinels, the valid first allele), totals, the per-read side path
// for rare alleles (N, -, _), the tile flush, L2 prefetch, the mbarrier arrive / back-off wait, and on the host the
// launch of the persistent kernels.
#pragma once
#include <type_traits>

#include "hx_internal.cuh"

namespace {

__device__ __forceinline__ unsigned long long warp_sum_ull(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-level accumulation of the four ingestion totals into global memory.
__device__ __forceinline__ void flush_totals(unsigned long long t0, unsigned long long t1,
                                             unsigned long long t2, unsigned long long t3,
                                             unsigned long long *totals) {
    __shared__ unsigned long long sh[4];
    if (threadIdx.x < 4) sh[threadIdx.x] = 0;
    __syncthreads();
    t0 = warp_sum_ull(t0); t1 = warp_sum_ull(t1); t2 = warp_sum_ull(t2); t3 = warp_sum_ull(t3);
    if ((threadIdx.x & 31) == 0) {
        if (t0) atomicAdd(&sh[0], t0);
        if (t1) atomicAdd(&sh[1], t1);
        if (t2) atomicAdd(&sh[2], t2);
        if (t3) atomicAdd(&sh[3], t3);
    }
    __syncthreads();
    if (threadIdx.x < 4 && sh[threadIdx.x]) atomicAdd(&totals[threadIdx.x], sh[threadIdx.x]);
}

__device__ __forceinline__ bool sym_valid_from(unsigned a) {   // util.py:258
    return a != HX_SYM_N && a != HX_SYM_GAP && a <= 6;
}

// A read of k >= 2 SNPs (fewer are skipped, util.py:230) at rank r must lie in [0, N] and fit the band (k <= W + 1);
// any other is an HX_E_READ error (bit 1).
__device__ __forceinline__ bool read_fits(int r, int64_t k, int N, int W) {
    return !(r < 0 || (int64_t)r + k > N || k - 1 > W);
}

// The start sentinel (util.py:262-266) and the end sentinel (:271-275) of a valid read of k >= 2 SNPs at rank r with
// codes c and first code a0 = c[0]; a read of two SNPs that is both first and last gets only the start one.  Adds the
// increments it made to n_sent (the counter is updated in place: returning them cost k_lr_transpose 7 registers).
template <class Count>
__device__ __forceinline__ void add_sentinels(const uint8_t *__restrict__ c, unsigned a0, int r, int k, int N,
                                              int64_t W, const HxCnt cnt, Count &n_sent) {
    if (r == 0 && sym_valid_from(a0)) {
        atomicAdd(cnt.cell(W, 0, 1) + HX_SYM_GAP * HX_NSYM + a0, 1u);
        n_sent++;
    }
    if (r + k == N && !(k == 2 && r == 0)) {
        const unsigned ap = c[k - 2], bl = c[k - 1];
        if (sym_valid_from(ap) && bl <= 6) {
            atomicAdd(cnt.cell(W, N, N + 1) + bl * HX_NSYM + HX_SYM_GAP, 1u);
            n_sent++;
        }
    }
}


// A read that holds N, - or _ : the pairs with such an allele on either side are not in the
// bit-planes; the whole warp adds them with REDs (lanes over the read's positions).
template <bool HI = true>   // HI = false: reads of at most 32 SNPs (one allele per lane)
__device__ __forceinline__ void bs_rare_read(const uint8_t *__restrict__ c, int kb, int r, int64_t W,
                                             const HxCnt cnt, unsigned &crumbs, unsigned &notcov,
                                             unsigned &errbits) {
    const int lane = threadIdx.x & 31;
    const unsigned a_lo = lane < kb ? c[lane] : 0xffu;
    const unsigned a_hi = HI && lane + 32 < kb ? c[lane + 32] : 0xffu;
    const unsigned m_lo = __ballot_sync(0xffffffffu, a_lo >= 4 && a_lo != 0xffu);
    const unsigned m_hi = HI ? __ballot_sync(0xffffffffu, a_hi >= 4 && a_hi != 0xffu) : 0u;
#pragma unroll
    for (int half = 0; half < (HI ? 2 : 1); ++half) {
        unsigned m = half ? m_hi : m_lo;
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const unsigned ai = __shfl_sync(0xffffffffu, half ? a_hi : a_lo, src);
            const int i = src + 32 * half;
            if (ai > 6) { errbits |= 2; continue; }
            if (lane == 0 && (ai == HX_SYM_N || ai == HX_SYM_GAP)) notcov++;
#pragma unroll
            for (int h2 = 0; h2 < (HI ? 2 : 1); ++h2) {
                const int j = lane + 32 * h2;
                const unsigned aj = h2 ? a_hi : a_lo;
                if (j >= kb || aj > 6) continue;
                if (j > i && ai == HX_SYM_DEL) {                 // '-' is a valid first allele
                    atomicAdd(cnt.cell(W, r + i + 1, r + j + 1) + ai * HX_NSYM + aj, 1u);
                    crumbs++;
                } else if (j < i && aj < 4) {                    // common first allele, rare second
                    atomicAdd(cnt.cell(W, r + j + 1, r + i + 1) + aj * HX_NSYM + ai, 1u);
                    crumbs++;
                }
            }
        }
    }
}


// Rows [pj_lo, pj_hi] of a sliding tile (ring of `rows` band rows of cells x 16 counters, row = pj % rows, cell = d-1,
// 16 = (a,b) in ACGT x ACGT), by the nthreads threads that call it: adds every non-zero counter to HBM and, with
// zero, clears it; returns the sum flushed by this thread (every regular-cell increment is one crumb,
// util.py:268,276,281).
__device__ __forceinline__ unsigned long long bs_flush_rows(uint32_t *tile32, int rows, int cells, int64_t pj_lo,
                                                            int64_t pj_hi, int64_t W, const HxCnt cnt, unsigned nthreads,
                                                            bool zero) {
    unsigned long long sum = 0;
    const int per_row = cells * 16;
    int row = (int)(pj_lo % rows);
    for (int64_t pj = pj_lo; pj <= pj_hi; ++pj) {
        uint32_t *base = tile32 + (size_t)row * per_row;
        for (int w = threadIdx.x; w < per_row; w += nthreads) {
            const uint32_t v = base[w];
            if (v) {
                const int d = (w >> 4) + 1, ab = w & 15;
                atomicAdd(cnt.cell(W, pj - d, pj) + (ab >> 2) * HX_NSYM + (ab & 3), v);
                if (zero) base[w] = 0;
                sum += v;
            }
        }
        if (++row == rows) row = 0;
    }
    return sum;
}


// L2 prefetch of the inputs of the batch after the one being transposed (TMA prefetch, no destination):
// the packed reads are streamed from HBM exactly once, so without it every group build pays two
// dependent HBM misses (offsets, then codes).
__device__ __forceinline__ void bs_prefetch_l2(const void *p, uint32_t bytes) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)15;
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a), "r"((bytes + 31u) & ~15u) : "memory");
}


// The CTA's slice [lo, hi) of rank-sorted reads: equal shares of the weight
//   f(i) = alleles before read i + HX_SLICE_READ_W * i + HX_SLICE_RANK_W * (rank[i] - rank[0])
// - the per-allele, per-read and per-run costs of the sorted-run kernels - not of the read count: SNP density varies
// along a region and with it the alleles per read and the runs per read (BASELINE configs[2]: the densest of 148
// equal-count slices holds 1.34x the mean).  Slice c starts at the first i with f(i) >= total * c / grid; warps 0 and 1
// find the two ends with a 32-ary search over off[] / rank[].  Every thread of the CTA must call it (one barrier).
constexpr int HX_SLICE_READ_W = 16, HX_SLICE_RANK_W = 8192;      // swept on the B200 with k1_umma on configs[2]
__device__ __forceinline__ void hx_weighted_slice(const int32_t *__restrict__ rank, const int64_t *__restrict__ off,
                                                  int64_t n_reads, int read_w, int rank_w, int64_t &lo, int64_t &hi) {
    __shared__ long long s_lohi[2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (warp < 2) {
        const int64_t base = off[0];
        const int64_t rbase = rank[0];
        const int64_t total = off[n_reads] - base + (int64_t)read_w * n_reads + (int64_t)rank_w * (rank[n_reads - 1] - rbase);
        const int c = (int)blockIdx.x + warp;
        const int64_t G = (int64_t)gridDim.x;
        const int64_t target = c >= (int)gridDim.x ? total : (total / G) * c + ((total % G) * c) / G;
        int64_t a = 0, b = n_reads;                      // the answer lies in [a, b]: f(n_reads) = total >= target
        while (a < b) {
            const int64_t span = b - a;
            const int64_t p = a + (span * (lane + 1)) / 33;               // 32 probes inside [a, b)
            const bool ge = off[p] - base + (int64_t)read_w * p + (int64_t)rank_w * (rank[p] - rbase) >= target;
            const unsigned m = __ballot_sync(0xffffffffu, ge);
            if (m == 0) {
                a = __shfl_sync(0xffffffffu, p, 31) + 1;
            } else {
                const int first = __ffs(m) - 1;
                b = __shfl_sync(0xffffffffu, p, first);
                if (first > 0) a = __shfl_sync(0xffffffffu, p, first - 1) + 1;
            }
        }
        if (lane == 0) s_lohi[warp] = a;
    }
    __syncthreads();
    lo = s_lohi[0];
    hi = s_lohi[1];
}

__device__ __forceinline__ void ws_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// hx_mbar_wait with a back-off between polls: for waits that normally last microseconds (many warps waiting)
__device__ __forceinline__ void ws_mbar_wait_sleep(uint32_t bar, uint32_t parity) {
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) break;
        __nanosleep(200);
    }
}
__device__ __forceinline__ void ws_pair_barrier(int nthreads) {
    asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}


// ---- host --------------------------------------------------------------------------------------------------

// SMs the persistent ingestion kernels may use: all of the device's, or fewer when the matrix is told so (ingest_sms).
inline int ingest_sm_budget(const hx_matrix *h) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    if (h->use.ingest_sms > 0 && h->use.ingest_sms < sms) sms = h->use.ingest_sms;
    return sms;
}

// The instantiation of a kernel templated on FUSED that serves this matrix: pick(std::true_type) when its counts go
// to the GPUs of the fused multi-GPU exchange, pick(std::false_type) otherwise (see HxCnt::for_build).
template <class Pick>
auto ingest_kernel_for(const hx_matrix *h, Pick pick) {
    return h->peer_world > 1 ? pick(std::true_type{}) : pick(std::false_type{});
}

// Prepares a persistent ingestion kernel for a launch with `block` threads and `smem` bytes of dynamic shared memory
// and sets *grid: one CTA per SM of the budget (with `occupancy`, as many as fit on an SM), but no CTA thinner than
// 256 reads.
template <class Kern>
int ingest_grid(Kern kern, int sms, int block, size_t smem, bool occupancy, int64_t n_reads, unsigned *grid) {
    HX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 1;
    if (occupancy) {
        HX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, block, smem));
        if (occ < 1) occ = 1;
    }
    const int64_t max_useful = (n_reads + 255) / 256;
    *grid = (unsigned)std::min((int64_t)sms * occ, max_useful);
    return HX_OK;
}


}  // namespace
