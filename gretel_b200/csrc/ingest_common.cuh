// Device helpers shared by the ingestion kernels (ingest.cu, ingest_umma.cu): totals, the per-read side path
// for rare alleles (N, -, _), L2 prefetch and the mbarrier arrive / back-off wait.
#pragma once
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


}  // namespace
