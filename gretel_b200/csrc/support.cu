// Read support for recovered haplotypes (hx_assign_reads): every packed read against every haplotype, by
// mismatches at the read's informative sites (codes other than N and _).  The read goes to the haplotypes with
// the fewest mismatches; ties split the read equally, in 32.32 fixed point, so every output is an integer and
// independent of the order in which reads are summed.  The definition is in DESIGN.md ("Read support").
//
// Bit planes: a code is 3 bits, so a haplotype is three bit-planes with 32 sites per word, and the mismatches of
// 32 sites are popc(valid & ((r0^p0)|(r1^p1)|(r2^p2))).  One thread per read builds the read's planes and shifts
// the haplotype words to the read's first site with a funnel shift.
#include <limits.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "hx_internal.cuh"

namespace {

constexpr int SUP_THREADS = 256;
constexpr int SUP_SMEM_HAPS = 2048;          // haplotypes whose per-CTA sums live in shared memory; the rest go to global
constexpr int64_t SUP_CHUNK_READS = 1 << 20; // reads per chunk: bounds the device scratch
constexpr int64_t SUP_CHUNK_CODES = 1 << 26;
constexpr int SUP_ERR_RANGE = 1, SUP_ERR_CODE = 2, SUP_ERR_HAP = 4;

// Device sums, one uint64 array: unique[H], shared[H], share_q32[H], then assigned, uninformative, over_limit and
// the error bits.
struct SupSums {
    unsigned long long *unique, *shared, *share, *totals, *err;
    __host__ __device__ SupSums(unsigned long long *base, int H)
        : unique(base), shared(base + H), share(base + 2 * (int64_t)H), totals(base + 3 * (int64_t)H),
          err(base + 3 * (int64_t)H + 3) {}
};

__host__ __device__ __forceinline__ int64_t plane_words(int N) { return (int64_t)(N >> 5) + 2; }

// planes[h][w] = {bit 0, bit 1, bit 2 of the codes of sites 32w..32w+31, 0}; sites past N are 0
__global__ void k_hap_planes(const uint8_t *__restrict__ haps, int H, int N, uint4 *__restrict__ planes,
                             unsigned long long *__restrict__ err) {
    const int64_t nw = plane_words(N);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)H * nw) return;
    const int64_t h = i / nw, w = i - h * nw;
    const uint8_t *hap = haps + h * ((int64_t)N + 1);
    uint32_t p0 = 0, p1 = 0, p2 = 0;
    bool bad = false;
    for (int b = 0; b < 32; ++b) {
        const int64_t s = w * 32 + b;
        if (s > N) break;
        const uint32_t c = hap[s];
        bad |= s >= 1 && c > 6;
        p0 |= (c & 1u) << b;
        p1 |= (c >> 1 & 1u) << b;
        p2 |= (c >> 2 & 1u) << b;
    }
    planes[i] = make_uint4(p0, p1, p2, 0u);
    if (bad) atomicOr(err, (unsigned long long)SUP_ERR_HAP);
}

struct ReadChunk {
    uint32_t r0, r1, r2, valid;
    bool bad;                        // a code > 6
};

// the read's planes for sites s..s+n-1 (n <= 32) from codes c[0..n-1]
__device__ __forceinline__ ReadChunk read_chunk(const uint8_t *__restrict__ c, int n) {
    ReadChunk q{0u, 0u, 0u, 0u, false};
#pragma unroll 1                     // unrolled, this loop makes k_assign_reads spill to local memory
    for (int b = 0; b < n; ++b) {
        const uint32_t x = c[b];
        q.bad |= x > 6;
        q.r0 |= (x & 1u) << b;
        q.r1 |= (x >> 1 & 1u) << b;
        q.r2 |= (x >> 2 & 1u) << b;
    }
    // N (100) and _ (110) are the codes with bit 2 set and bit 0 clear
    q.valid = ~(q.r2 & ~q.r0) & (n == 32 ? 0xffffffffu : ((1u << n) - 1u));
    return q;
}

// mismatches between a read chunk starting at site s and haplotype planes hp (of one haplotype)
__device__ __forceinline__ int chunk_mismatches(const ReadChunk &q, const uint4 *__restrict__ hp, int64_t s) {
    const uint4 lo = hp[s >> 5], hi = hp[(s >> 5) + 1];
    const uint32_t sh = (uint32_t)(s & 31);
    const uint32_t h0 = __funnelshift_r(lo.x, hi.x, sh), h1 = __funnelshift_r(lo.y, hi.y, sh),
                   h2 = __funnelshift_r(lo.z, hi.z, sh);
    return __popc(q.valid & ((q.r0 ^ h0) | (q.r1 ^ h1) | (q.r2 ^ h2)));
}

// d_h of a read of k > 32 sites from site s0 on: the chunks are rebuilt for every haplotype (long reads only)
__device__ __forceinline__ int long_mismatches(const uint8_t *__restrict__ c, int64_t k, int64_t s0,
                                               const uint4 *__restrict__ hp) {
    int d = 0;
    for (int64_t t = 0; t < k; t += 32) {
        const ReadChunk q = read_chunk(c + t, (int)(k - t < 32 ? k - t : 32));
        d += chunk_mismatches(q, hp, s0 + t);
    }
    return d;
}

__global__ void __launch_bounds__(SUP_THREADS)
k_assign_reads(const int32_t *__restrict__ rank, const int64_t *__restrict__ off, const uint8_t *__restrict__ codes,
               int64_t n_reads, const uint4 *__restrict__ planes, int H, int N, int max_mismatch,
               unsigned long long *__restrict__ sums, int32_t *__restrict__ best_mm, int32_t *__restrict__ n_best,
               int32_t *__restrict__ first_best) {
    extern __shared__ unsigned long long s_mem[];
    const int hs = min(H, SUP_SMEM_HAPS);
    unsigned long long *s_share = s_mem;                               // [hs]
    unsigned *s_unique = reinterpret_cast<unsigned *>(s_mem + hs);     // [hs]
    unsigned *s_shared = s_unique + hs;                                // [hs]
    __shared__ unsigned s_tot[3];
    __shared__ unsigned s_err;
    for (int i = threadIdx.x; i < hs; i += blockDim.x) { s_share[i] = 0; s_unique[i] = 0; s_shared[i] = 0; }
    if (threadIdx.x < 3) s_tot[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_err = 0;
    __syncthreads();
    const SupSums g(sums, H);
    const int64_t nw = plane_words(N);

    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_reads; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = rank[i], k = off[i + 1] - off[i];
        if (r < 0 || k < 0 || r + k > N) {
            atomicOr(&s_err, (unsigned)SUP_ERR_RANGE);
            continue;
        }
        const uint8_t *c = codes + off[i];
        const int64_t s0 = r + 1;
        // informative sites and code checks; the planes of a read of <= 32 sites are kept for the haplotype loop
        bool bad = false;
        int m = 0;
        ReadChunk q0{0u, 0u, 0u, 0u, false};
        for (int64_t t = 0; t < k; t += 32) {
            const ReadChunk q = read_chunk(c + t, (int)(k - t < 32 ? k - t : 32));
            bad |= q.bad;
            m += __popc(q.valid);
            if (t == 0) q0 = q;
        }
        if (bad) {
            atomicOr(&s_err, (unsigned)SUP_ERR_CODE);
            continue;
        }
        int D = INT_MAX, nb = 0, first = -1;
        if (m > 0) {
            for (int h = 0; h < H; ++h) {
                const uint4 *hp = planes + h * nw;
                const int d = k <= 32 ? chunk_mismatches(q0, hp, s0) : long_mismatches(c, k, s0, hp);
                if (d < D) { D = d; nb = 1; first = h; }
                else if (d == D) ++nb;
            }
        }
        const int status = m == 0 ? 1 : (max_mismatch >= 0 && D > max_mismatch) ? 2 : 0;   // totals slot
        atomicAdd(&s_tot[status], 1u);
        if (best_mm) {
            best_mm[i] = m == 0 ? -1 : D;
            n_best[i] = m == 0 ? 0 : nb;
            first_best[i] = status == 0 ? first : -1;
        }
        if (status != 0) continue;
        if (nb == 1) {
            if (first < hs) { atomicAdd(&s_unique[first], 1u); atomicAdd(&s_share[first], 1ull << 32); }
            else { atomicAdd(&g.unique[first], 1ull); atomicAdd(&g.share[first], 1ull << 32); }
            continue;
        }
        // a tie: find the tied set again (a per-read mask of H bits would be unbounded)
        const unsigned long long q32 = (1ull << 32) / (unsigned)nb;
        int left = nb;
        for (int h = first; left > 0; ++h) {
            const uint4 *hp = planes + h * nw;
            const int d = k <= 32 ? chunk_mismatches(q0, hp, s0) : long_mismatches(c, k, s0, hp);
            if (d != D) continue;
            --left;
            if (h < hs) { atomicAdd(&s_shared[h], 1u); atomicAdd(&s_share[h], q32); }
            else { atomicAdd(&g.shared[h], 1ull); atomicAdd(&g.share[h], q32); }
        }
    }
    __syncthreads();
    for (int h = threadIdx.x; h < hs; h += blockDim.x) {
        if (s_unique[h]) atomicAdd(&g.unique[h], (unsigned long long)s_unique[h]);
        if (s_shared[h]) atomicAdd(&g.shared[h], (unsigned long long)s_shared[h]);
        if (s_share[h]) atomicAdd(&g.share[h], s_share[h]);
    }
    if (threadIdx.x < 3 && s_tot[threadIdx.x]) atomicAdd(&g.totals[threadIdx.x], (unsigned long long)s_tot[threadIdx.x]);
    if (threadIdx.x == 0 && s_err) atomicOr(g.err, (unsigned long long)s_err);
}

}  // namespace

// Device time of one kernel launch on the matrix's stream, added to the assignment timer.
template <class Launch>
static int timed(hx_matrix *h, Launch launch) {
    HX_CUDA(cudaEventRecord(h->a_ev[0], h->stream));
    launch();
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    HX_CUDA(cudaEventRecord(h->a_ev[1], h->stream));
    HX_CUDA(cudaEventSynchronize(h->a_ev[1]));
    float ms = 0.0f;
    HX_CUDA(cudaEventElapsedTime(&ms, h->a_ev[0], h->a_ev[1]));
    h->use.last_ms[3] += ms;
    return HX_OK;
}

void hx_support_free(hx_matrix *h) {
    cudaStream_t st = h->stream;
    h->a_haps.release(st); h->a_planes.release(st); h->a_sums.release(st);
    h->a_rank.release(st); h->a_off.release(st); h->a_codes.release(st); h->a_best.release(st);
    for (int e = 0; e < 2; ++e) {
        if (h->a_ev[e]) cudaEventDestroy(h->a_ev[e]);
        h->a_ev[e] = nullptr;
    }
}

extern "C" int hx_assign_reads(hx_matrix *h, const uint8_t *haps, int32_t n_haps, const int32_t *rank,
                               const int64_t *off, const uint8_t *codes, int64_t n_reads, int32_t max_mismatch,
                               int64_t *unique, int64_t *shared, uint64_t *share_q32, int64_t totals[3],
                               int32_t *best_mm, int32_t *n_best, int32_t *first_best) {
    HX_CHECK_ARG(h && haps && n_haps >= 1 && n_reads >= 0 && unique && shared && share_q32 && totals);
    HX_CHECK_ARG(n_reads == 0 || (rank && off && codes));
    const bool per_read = best_mm || n_best || first_best;
    HX_CHECK_ARG(!per_read || (best_mm && n_best && first_best));
    HX_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int N = h->N, H = n_haps;
    const int64_t nw = plane_words(N), n_sums = 3 * (int64_t)H + 4;
    for (int e = 0; e < 2; ++e)
        if (!h->a_ev[e]) HX_CUDA(cudaEventCreate(&h->a_ev[e]));
    h->use.last_ms[3] = 0.0f;

    HX_CUDA(h->a_haps.grow((int64_t)H * (N + 1), st));
    HX_CUDA(h->a_planes.grow(sizeof(uint4) * H * nw, st));
    HX_CUDA(h->a_sums.grow(sizeof(unsigned long long) * n_sums, st));
    HX_CUDA(hx_fill_async(h->a_sums.p, 0, sizeof(unsigned long long) * n_sums, st));
    HX_CUDA(cudaMemcpyAsync(h->a_haps.p, haps, (size_t)H * (N + 1), cudaMemcpyHostToDevice, st));
    const int64_t n_planes = (int64_t)H * nw;
    int rc = timed(h, [&] {
        k_hap_planes<<<(unsigned)((n_planes + 255) / 256), 256, 0, st>>>(h->a_haps.p, H, N, h->a_planes.p,
                                                                        SupSums(h->a_sums.p, H).err);
    });
    if (rc) return rc;

    int sms = 148;
    HX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
    const int hs = std::min(H, SUP_SMEM_HAPS);
    const size_t smem = (size_t)hs * (sizeof(unsigned long long) + 2 * sizeof(unsigned));
    // reads in chunks at read boundaries, at most SUP_CHUNK_READS reads and about SUP_CHUNK_CODES codes each
    for (int64_t a = 0; a < n_reads;) {
        int64_t b = std::min(n_reads, a + SUP_CHUNK_READS);
        if (off[b] - off[a] > SUP_CHUNK_CODES)
            b = std::max(a + 1, (int64_t)(std::upper_bound(off + a, off + b + 1, off[a] + SUP_CHUNK_CODES) - off) - 1);
        const int64_t nr = b - a, nc = off[b] - off[a];
        HX_CHECK_ARG(nc >= 0);
        HX_CUDA(h->a_rank.grow(sizeof(int32_t) * nr, st));
        HX_CUDA(h->a_off.grow(sizeof(int64_t) * (nr + 1), st));
        HX_CUDA(h->a_codes.grow(nc + 16, st));
        if (per_read) HX_CUDA(h->a_best.grow(sizeof(int32_t) * 3 * nr, st));
        HX_CUDA(cudaMemcpyAsync(h->a_rank.p, rank + a, sizeof(int32_t) * nr, cudaMemcpyHostToDevice, st));
        HX_CUDA(cudaMemcpyAsync(h->a_off.p, off + a, sizeof(int64_t) * (nr + 1), cudaMemcpyHostToDevice, st));
        if (nc) HX_CUDA(cudaMemcpyAsync(h->a_codes.p, codes + off[a], (size_t)nc, cudaMemcpyHostToDevice, st));
        int32_t *d_best = per_read ? h->a_best.p : nullptr;
        const int64_t want = (nr + SUP_THREADS - 1) / SUP_THREADS;
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)sms * 4));
        rc = timed(h, [&] {
            // the kernel indexes codes by absolute offsets: bias the base pointer by off[a]
            k_assign_reads<<<grid, SUP_THREADS, smem, st>>>(
                h->a_rank.p, h->a_off.p, h->a_codes.p - off[a], nr, h->a_planes.p, H, N, max_mismatch, h->a_sums.p,
                d_best, d_best ? d_best + nr : nullptr, d_best ? d_best + 2 * nr : nullptr);
        });
        if (rc) return rc;
        if (per_read) {
            HX_CUDA(cudaMemcpyAsync(best_mm + a, d_best, sizeof(int32_t) * nr, cudaMemcpyDeviceToHost, st));
            HX_CUDA(cudaMemcpyAsync(n_best + a, d_best + nr, sizeof(int32_t) * nr, cudaMemcpyDeviceToHost, st));
            HX_CUDA(cudaMemcpyAsync(first_best + a, d_best + 2 * nr, sizeof(int32_t) * nr, cudaMemcpyDeviceToHost, st));
        }
        a = b;
    }

    unsigned long long *hs_sums = (unsigned long long *)malloc(sizeof(unsigned long long) * n_sums);
    if (!hs_sums) return HX_E_NOMEM;
    const cudaError_t e1 = cudaMemcpyAsync(hs_sums, h->a_sums.p, sizeof(unsigned long long) * n_sums,
                                           cudaMemcpyDeviceToHost, st);
    const cudaError_t e2 = e1 == cudaSuccess ? cudaStreamSynchronize(st) : e1;
    if (e2 != cudaSuccess) {
        free(hs_sums);
        HX_CUDA(e2);
    }
    const SupSums s(hs_sums, H);
    const unsigned long long err = *s.err;
    for (int i = 0; i < H; ++i) {
        unique[i] = (int64_t)s.unique[i];
        shared[i] = (int64_t)s.shared[i];
        share_q32[i] = s.share[i];
    }
    for (int i = 0; i < 3; ++i) totals[i] = (int64_t)s.totals[i];
    free(hs_sums);
    if (err & SUP_ERR_HAP) {
        hx_set_error("hx_assign_reads: haplotype code > 6 at a site in 1..N");
        return HX_E_ARG;
    }
    if (err) {
        hx_set_error("hx_assign_reads: invalid packed read(s): %s%s",
                     (err & SUP_ERR_RANGE) ? "[read leaves [1,N]] " : "", (err & SUP_ERR_CODE) ? "[allele code > 6]" : "");
        return HX_E_READ;
    }
    return HX_OK;
}
