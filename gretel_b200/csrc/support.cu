// Read support for recovered haplotypes (hx_assign_reads): every packed read against every haplotype, by
// mismatches at the read's informative sites (codes other than N and _).  The read goes to the haplotypes with
// the fewest mismatches; ties split the read equally, in 32.32 fixed point, so every output is an integer and
// independent of the order in which reads are summed.  The definition is in DESIGN.md ("Read support").  The
// compatibility classes of the reads (hx_read_classes: reads grouped by their set of best haplotypes) and the EM over
// them that estimates each haplotype's abundance (hx_em_abundance, host code) are DESIGN.md §4 K7.
//
// Bit planes: a code is 3 bits, so a haplotype is three bit-planes with 32 sites per word, and the mismatches of
// 32 sites are popc(valid & ((r0^p0)|(r1^p1)|(r2^p2))).  One thread per read builds the read's planes and shifts
// the haplotype words to the read's first site with a funnel shift.
#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <new>
#include <vector>

#include "hx_internal.cuh"
#include "scan.cuh"

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

// What the scan of one read finds (DESIGN.md §4 K5): its informative sites m, the fewest mismatches D, the number of
// haplotypes nb at D and the lowest of them, and its totals slot.  err != 0: the read is invalid and nothing else is
// set.  The planes of a read of <= 32 sites are kept in q0 for a second pass over the haplotypes.
struct ReadScan {
    const uint8_t *c;
    int64_t k, s0;
    ReadChunk q0;
    int m, D, nb, first, status;     // status: 0 assigned, 1 uninformative, 2 over the limit
    unsigned err;
};

// d_h of the scanned read against haplotype planes hp
__device__ __forceinline__ int scan_mismatches(const ReadScan &x, const uint4 *__restrict__ hp) {
    return x.k <= 32 ? chunk_mismatches(x.q0, hp, x.s0) : long_mismatches(x.c, x.k, x.s0, hp);
}

// the per-read scan that read support (k_assign_reads) and read classes (k_class_scan) share
__device__ __forceinline__ ReadScan scan_read(const int32_t *__restrict__ rank, const int64_t *__restrict__ off,
                                              const uint8_t *__restrict__ codes, int64_t i,
                                              const uint4 *__restrict__ planes, int H, int N, int max_mismatch) {
    ReadScan x;
    x.err = 0;
    const int64_t r = rank[i];
    x.k = off[i + 1] - off[i];
    if (r < 0 || x.k < 0 || r + x.k > N) {
        x.err = SUP_ERR_RANGE;
        return x;
    }
    x.c = codes + off[i];
    x.s0 = r + 1;
    // informative sites and code checks
    bool bad = false;
    x.m = 0;
    x.q0 = ReadChunk{0u, 0u, 0u, 0u, false};
    for (int64_t t = 0; t < x.k; t += 32) {
        const ReadChunk q = read_chunk(x.c + t, (int)(x.k - t < 32 ? x.k - t : 32));
        bad |= q.bad;
        x.m += __popc(q.valid);
        if (t == 0) x.q0 = q;
    }
    if (bad) {
        x.err = SUP_ERR_CODE;
        return x;
    }
    const int64_t nw = plane_words(N);
    x.D = INT_MAX; x.nb = 0; x.first = -1;
    if (x.m > 0) {
        for (int h = 0; h < H; ++h) {
            const int d = scan_mismatches(x, planes + h * nw);
            if (d < x.D) { x.D = d; x.nb = 1; x.first = h; }
            else if (d == x.D) ++x.nb;
        }
    }
    x.status = x.m == 0 ? 1 : (max_mismatch >= 0 && x.D > max_mismatch) ? 2 : 0;
    return x;
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
        const ReadScan x = scan_read(rank, off, codes, i, planes, H, N, max_mismatch);
        if (x.err) {
            atomicOr(&s_err, x.err);
            continue;
        }
        const int D = x.D, nb = x.nb, first = x.first, status = x.status;
        atomicAdd(&s_tot[status], 1u);
        if (best_mm) {
            best_mm[i] = x.m == 0 ? -1 : D;
            n_best[i] = x.m == 0 ? 0 : nb;
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
            if (scan_mismatches(x, planes + h * nw) != D) continue;
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

// ---- read classes (DESIGN.md §4 K7) --------------------------------------------------------------------------------
// An assigned read belongs to the class keyed by its tie set B.  Singletons are counted per haplotype, as K5 counts
// unique[h].  A tied read writes nb = |B| (0 for every other read) and (first, D), so that its members can be
// enumerated again after the scan of nb has placed them in the member pool.
__global__ void __launch_bounds__(SUP_THREADS)
k_class_scan(const int32_t *__restrict__ rank, const int64_t *__restrict__ off, const uint8_t *__restrict__ codes,
             int64_t n_reads, const uint4 *__restrict__ planes, int H, int N, int max_mismatch,
             unsigned long long *__restrict__ sums, int64_t *__restrict__ nb_out, int2 *__restrict__ tie) {
    extern __shared__ unsigned long long s_mem[];
    const int hs = min(H, SUP_SMEM_HAPS);
    unsigned *s_unique = reinterpret_cast<unsigned *>(s_mem);         // [hs]
    __shared__ unsigned s_tot[3];
    __shared__ unsigned s_err;
    for (int i = threadIdx.x; i < hs; i += blockDim.x) s_unique[i] = 0;
    if (threadIdx.x < 3) s_tot[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_err = 0;
    __syncthreads();
    const SupSums g(sums, H);

    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_reads; i += (int64_t)gridDim.x * blockDim.x) {
        const ReadScan x = scan_read(rank, off, codes, i, planes, H, N, max_mismatch);
        int64_t nb = 0;
        if (x.err) {
            atomicOr(&s_err, x.err);
        } else {
            atomicAdd(&s_tot[x.status], 1u);
            if (x.status == 0 && x.nb == 1) {
                if (x.first < hs) atomicAdd(&s_unique[x.first], 1u);
                else atomicAdd(&g.unique[x.first], 1ull);
            } else if (x.status == 0) {
                nb = x.nb;
                tie[i] = make_int2(x.first, x.D);
            }
        }
        nb_out[i] = nb;
    }
    __syncthreads();
    for (int h = threadIdx.x; h < hs; h += blockDim.x)
        if (s_unique[h]) atomicAdd(&g.unique[h], (unsigned long long)s_unique[h]);
    if (threadIdx.x < 3 && s_tot[threadIdx.x]) atomicAdd(&g.totals[threadIdx.x], (unsigned long long)s_tot[threadIdx.x]);
    if (threadIdx.x == 0 && s_err) atomicOr(g.err, (unsigned long long)s_err);
}

// 64-bit FNV-1a step over a member index, and the final mix that spreads it over the table
__device__ __forceinline__ unsigned long long fnv_step(unsigned long long x, int h) {
    return (x ^ (unsigned long long)(unsigned)h) * 0x100000001b3ull;
}
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    return x;
}

// Tied reads [lo, hi) of the chunk: B ascending into pool[moff[i] - base ..], and the hash of B masked by hash_mask.
__global__ void __launch_bounds__(SUP_THREADS)
k_class_members(const int32_t *__restrict__ rank, const int64_t *__restrict__ off, const uint8_t *__restrict__ codes,
                int64_t lo, int64_t hi, const uint4 *__restrict__ planes, int N, const int64_t *__restrict__ nb,
                const int2 *__restrict__ tie, const int64_t *__restrict__ moff, int64_t base,
                int32_t *__restrict__ pool, unsigned long long *__restrict__ hash, unsigned long long hash_mask) {
    const int64_t nw = plane_words(N);
    for (int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (int64_t)gridDim.x * blockDim.x) {
        const int n = (int)nb[i];
        if (n == 0) continue;
        ReadScan x{};                                // a valid assigned read: only its planes are needed again
        x.k = off[i + 1] - off[i];
        x.c = codes + off[i];
        x.s0 = (int64_t)rank[i] + 1;
        if (x.k <= 32) x.q0 = read_chunk(x.c, (int)x.k);
        const int2 fd = tie[i];
        int32_t *out = pool + (moff[i] - base);
        unsigned long long hv = 0xcbf29ce484222325ull;
        int j = 0;
        for (int h = fd.x; j < n; ++h) {
            if (scan_mismatches(x, planes + h * nw) != fd.y) continue;
            out[j++] = h;
            hv = fnv_step(hv, h);
        }
        hash[i] = mix64(hv) & hash_mask;
    }
}

// Tied reads [lo, hi) into an open-addressing table of S (a power of two) slots.  A slot holds a representative read,
// taken by CAS, and a count.  A read joins a slot only if the hash and the whole member list are equal; otherwise it
// probes on linearly.  No outcome depends on the hash being free of collisions.
__global__ void __launch_bounds__(SUP_THREADS)
k_class_insert(int64_t lo, int64_t hi, const int64_t *__restrict__ nb, const int64_t *__restrict__ moff, int64_t base,
               const int32_t *__restrict__ pool, const unsigned long long *__restrict__ hash, int32_t *slot_rep,
               unsigned *slot_cnt, uint32_t S) {
    for (int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t n = nb[i];
        if (n == 0) continue;
        const unsigned long long hv = hash[i];
        const int32_t *mine = pool + (moff[i] - base);
        for (uint32_t s = (uint32_t)mix64(hv) & (S - 1);; s = (s + 1) & (S - 1)) {
            const int32_t rep = atomicCAS(&slot_rep[s], -1, (int32_t)i);
            bool same = rep < 0;
            if (!same && hash[rep] == hv && nb[rep] == n) {
                const int32_t *theirs = pool + (moff[rep] - base);
                same = true;
                for (int64_t j = 0; j < n && same; ++j) same = theirs[j] == mine[j];
            }
            if (same) {
                atomicAdd(&slot_cnt[s], 1u);
                break;
            }
        }
    }
}

// Occupied slots to classes: cls[c] = {member position in out, |B|, count}, members copied to out.  ncls[0] counts
// the classes, ncls[1] the members; the order is whatever the atomics give (the host sorts).
__global__ void __launch_bounds__(SUP_THREADS)
k_class_compact(uint32_t S, const int32_t *__restrict__ slot_rep, const unsigned *__restrict__ slot_cnt,
                const int64_t *__restrict__ nb, const int64_t *__restrict__ moff, int64_t base,
                const int32_t *__restrict__ pool, unsigned long long *__restrict__ ncls, int4 *__restrict__ cls,
                int32_t *__restrict__ out) {
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < S; s += (int64_t)gridDim.x * blockDim.x) {
        const int32_t rep = slot_rep[s];
        if (rep < 0) continue;
        const int n = (int)nb[rep];
        const unsigned long long c = atomicAdd(&ncls[0], 1ull), p = atomicAdd(&ncls[1], (unsigned long long)n);
        cls[c] = make_int4((int)p, n, (int)slot_cnt[s], 0);
        const int32_t *src = pool + (moff[rep] - base);
        for (int j = 0; j < n; ++j) out[p + j] = src[j];
    }
}

}  // namespace

void hx_support_free(hx_matrix *h) {
    cudaStream_t st = h->stream;
    h->a_haps.release(st); h->a_planes.release(st); h->a_sums.release(st);
    h->a_rank.release(st); h->a_off.release(st); h->a_codes.release(st); h->a_best.release(st);
    h->cl_nb.release(st); h->cl_moff.release(st); h->cl_scan.release(st); h->cl_tie.release(st); h->cl_hash.release(st);
    h->cl_ncls.release(st); h->cl_pool.release(st); h->cl_rep.release(st); h->cl_out.release(st); h->cl_cnt.release(st);
    h->cl_cls.release(st);
    hx_classes_drop(h);
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
    int rc = timed(h, 3, [&] {
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
        rc = timed(h, 3, [&] {
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

// ---- read classes (DESIGN.md §4 K7) --------------------------------------------------------------------------------
// The classes of the last hx_read_classes, in lexicographic order of their member lists.
struct hx_classes {
    std::vector<int64_t> off, count;
    std::vector<int32_t> members;
};

namespace {
// device scratch per member of a sub-batch: the pool and the compacted copy (4 + 4 B), and up to two table slots of
// a representative and a count (8 B each); a table has at least 2 slots per tied read and tied reads have >= 2 members
constexpr int64_t CLS_BYTES_PER_MEMBER = 24;
constexpr int CLS_SCAN_ITEMS = 16;

unsigned long long class_hash_mask() {
    const char *e = getenv("HX_CLASS_HASH_BITS");
    const int bits = e ? std::max(0, std::min(64, atoi(e))) : 64;
    return bits >= 64 ? ~0ull : (1ull << bits) - 1;
}

int64_t class_batch_members() {
    const char *e = getenv("HX_CLASS_SCRATCH_MB");
    const double mb = e ? atof(e) : 256.0;
    return std::max<int64_t>(1, (int64_t)(mb * 1048576.0 / CLS_BYTES_PER_MEMBER));
}
}  // namespace

void hx_classes_drop(hx_matrix *h) {
    delete h->a_cls;
    h->a_cls = nullptr;
}

extern "C" int hx_read_classes(hx_matrix *h, const uint8_t *haps, int32_t n_haps, const int32_t *rank,
                               const int64_t *off, const uint8_t *codes, int64_t n_reads, int32_t max_mismatch,
                               int64_t totals[3], int64_t *n_classes, int64_t *n_members) {
    if (h) hx_classes_drop(h);                                 // a failed call leaves no classes
    HX_CHECK_ARG(h && haps && n_haps >= 1 && n_reads >= 0 && totals && n_classes && n_members);
    HX_CHECK_ARG(n_reads == 0 || (rank && off && codes));
    HX_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int N = h->N, H = n_haps;
    const int64_t nw = plane_words(N), n_sums = 3 * (int64_t)H + 4;
    for (int e = 0; e < 2; ++e)
        if (!h->a_ev[e]) HX_CUDA(cudaEventCreate(&h->a_ev[e]));
    h->use.last_ms[5] = 0.0f;
    const unsigned long long mask = class_hash_mask();
    const int64_t batch_cap = class_batch_members();

    HX_CUDA(h->a_haps.grow((int64_t)H * (N + 1), st));
    HX_CUDA(h->a_planes.grow(sizeof(uint4) * H * nw, st));
    HX_CUDA(h->a_sums.grow(sizeof(unsigned long long) * n_sums, st));
    HX_CUDA(hx_fill_async(h->a_sums.p, 0, sizeof(unsigned long long) * n_sums, st));
    HX_CUDA(cudaMemcpyAsync(h->a_haps.p, haps, (size_t)H * (N + 1), cudaMemcpyHostToDevice, st));
    const int64_t n_planes = (int64_t)H * nw;
    int rc = timed(h, 5, [&] {
        k_hap_planes<<<(unsigned)((n_planes + 255) / 256), 256, 0, st>>>(h->a_haps.p, H, N, h->a_planes.p,
                                                                        SupSums(h->a_sums.p, H).err);
    });
    if (rc) return rc;

    int sms = 148;
    HX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
    const unsigned fill_grid = (unsigned)sms * 4;
    auto grid_for = [&](int64_t n) {
        return (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + SUP_THREADS - 1) / SUP_THREADS, fill_grid));
    };
    const int hs = std::min(H, SUP_SMEM_HAPS);
    const size_t smem = (size_t)hs * sizeof(unsigned);
    std::map<std::vector<int32_t>, int64_t> merged;            // member list -> count, over all chunks
    std::vector<int64_t> moff_h;
    std::vector<int4> cls_h;
    std::vector<int32_t> mem_h;
    // reads in chunks at read boundaries, as hx_assign_reads sends them
    for (int64_t a = 0; a < n_reads;) {
        int64_t b = std::min(n_reads, a + SUP_CHUNK_READS);
        if (off[b] - off[a] > SUP_CHUNK_CODES)
            b = std::max(a + 1, (int64_t)(std::upper_bound(off + a, off + b + 1, off[a] + SUP_CHUNK_CODES) - off) - 1);
        const int64_t nr = b - a, nc = off[b] - off[a];
        HX_CHECK_ARG(nc >= 0);
        const int64_t nblk = (nr + 256 * CLS_SCAN_ITEMS - 1) / (256 * CLS_SCAN_ITEMS);
        HX_CUDA(h->a_rank.grow(sizeof(int32_t) * nr, st));
        HX_CUDA(h->a_off.grow(sizeof(int64_t) * (nr + 1), st));
        HX_CUDA(h->a_codes.grow(nc + 16, st));
        HX_CUDA(h->cl_nb.grow(sizeof(int64_t) * nr, st));
        HX_CUDA(h->cl_moff.grow(sizeof(int64_t) * nr, st));
        HX_CUDA(h->cl_scan.grow(sizeof(int64_t) * (nblk + 1), st));
        HX_CUDA(h->cl_tie.grow(sizeof(int2) * nr, st));
        HX_CUDA(h->cl_hash.grow(sizeof(unsigned long long) * nr, st));
        HX_CUDA(cudaMemcpyAsync(h->a_rank.p, rank + a, sizeof(int32_t) * nr, cudaMemcpyHostToDevice, st));
        HX_CUDA(cudaMemcpyAsync(h->a_off.p, off + a, sizeof(int64_t) * (nr + 1), cudaMemcpyHostToDevice, st));
        if (nc) HX_CUDA(cudaMemcpyAsync(h->a_codes.p, codes + off[a], (size_t)nc, cudaMemcpyHostToDevice, st));
        // the kernels index codes by absolute offsets: bias the base pointer by off[a]
        const uint8_t *d_codes = h->a_codes.p - off[a];
        rc = timed(h, 5, [&] {
            k_class_scan<<<grid_for(nr), SUP_THREADS, smem, st>>>(h->a_rank.p, h->a_off.p, d_codes, nr, h->a_planes.p,
                                                                  H, N, max_mismatch, h->a_sums.p, h->cl_nb.p,
                                                                  h->cl_tie.p);
        });
        if (rc) return rc;
        // member offsets: exclusive scan of nb; the total lands in cl_scan[nblk]
        rc = timed(h, 5, [&] {
            k_scan_partials<int64_t, 0, CLS_SCAN_ITEMS><<<(unsigned)nblk, 256, 0, st>>>(h->cl_nb.p, nr, h->cl_scan.p);
            k_scan_spine<int64_t, 0><<<1, 32, 0, st>>>(h->cl_scan.p, nblk, h->cl_scan.p + nblk);
            k_scan_apply<int64_t, 0, CLS_SCAN_ITEMS, true><<<(unsigned)nblk, 256, 0, st>>>(h->cl_nb.p, nr, h->cl_scan.p,
                                                                                         h->cl_moff.p);
            h->use.launches += 2;
        });
        if (rc) return rc;
        int64_t total = 0;
        HX_CUDA(cudaMemcpyAsync(&total, h->cl_scan.p + nblk, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        HX_CUDA(cudaStreamSynchronize(st));
        a = b;
        if (total == 0) continue;
        // sub-batches of tied reads cut at their member offsets, at most batch_cap members each (or one read)
        const bool split = total > batch_cap;
        if (split) {
            moff_h.resize(nr + 1);
            HX_CUDA(cudaMemcpyAsync(moff_h.data(), h->cl_moff.p, sizeof(int64_t) * nr, cudaMemcpyDeviceToHost, st));
            HX_CUDA(cudaStreamSynchronize(st));
            moff_h[nr] = total;
        }
        for (int64_t lo = 0; lo < nr;) {
            int64_t hi = nr;
            if (split) {
                hi = (int64_t)(std::upper_bound(moff_h.begin() + lo + 1, moff_h.end(), moff_h[lo] + batch_cap) -
                               moff_h.begin()) - 1;
                hi = std::max(hi, lo + 1);
            }
            const int64_t base = split ? moff_h[lo] : 0, members = split ? moff_h[hi] - base : total;
            if (members == 0) { lo = hi; continue; }
            uint32_t S = 2;
            while (S < (uint64_t)members) S <<= 1;
            const int64_t max_cls = members / 2;
            HX_CUDA(h->cl_pool.grow(sizeof(int32_t) * members, st));
            HX_CUDA(h->cl_out.grow(sizeof(int32_t) * members, st));
            HX_CUDA(h->cl_rep.grow(sizeof(int32_t) * S, st));
            HX_CUDA(h->cl_cnt.grow(sizeof(unsigned) * S, st));
            HX_CUDA(h->cl_cls.grow(sizeof(int4) * max_cls, st));
            HX_CUDA(h->cl_ncls.grow(sizeof(unsigned long long) * 2, st));
            HX_CUDA(hx_fill_async(h->cl_rep.p, 0xff, sizeof(int32_t) * S, st));
            HX_CUDA(hx_fill_async(h->cl_cnt.p, 0, sizeof(unsigned) * S, st));
            HX_CUDA(hx_fill_async(h->cl_ncls.p, 0, sizeof(unsigned long long) * 2, st));
            const int64_t n_lo = lo, n_hi = hi;
            rc = timed(h, 5, [&] {
                k_class_members<<<grid_for(n_hi - n_lo), SUP_THREADS, 0, st>>>(
                    h->a_rank.p, h->a_off.p, d_codes, n_lo, n_hi, h->a_planes.p, N, h->cl_nb.p, h->cl_tie.p,
                    h->cl_moff.p, base, h->cl_pool.p, h->cl_hash.p, mask);
                k_class_insert<<<grid_for(n_hi - n_lo), SUP_THREADS, 0, st>>>(
                    n_lo, n_hi, h->cl_nb.p, h->cl_moff.p, base, h->cl_pool.p, h->cl_hash.p, h->cl_rep.p, h->cl_cnt.p, S);
                k_class_compact<<<grid_for(S), SUP_THREADS, 0, st>>>(S, h->cl_rep.p, h->cl_cnt.p, h->cl_nb.p,
                                                                      h->cl_moff.p, base, h->cl_pool.p, h->cl_ncls.p,
                                                                      h->cl_cls.p, h->cl_out.p);
                h->use.launches += 2;
            });
            if (rc) return rc;
            unsigned long long ncls[2];
            HX_CUDA(cudaMemcpyAsync(ncls, h->cl_ncls.p, sizeof(ncls), cudaMemcpyDeviceToHost, st));
            HX_CUDA(cudaStreamSynchronize(st));
            cls_h.resize(ncls[0]);
            mem_h.resize(ncls[1]);
            HX_CUDA(cudaMemcpyAsync(cls_h.data(), h->cl_cls.p, sizeof(int4) * ncls[0], cudaMemcpyDeviceToHost, st));
            HX_CUDA(cudaMemcpyAsync(mem_h.data(), h->cl_out.p, sizeof(int32_t) * ncls[1], cudaMemcpyDeviceToHost, st));
            HX_CUDA(cudaStreamSynchronize(st));
            for (const int4 &c : cls_h)
                merged[std::vector<int32_t>(mem_h.begin() + c.x, mem_h.begin() + c.x + c.y)] += c.z;
            lo = hi;
        }
    }

    std::vector<unsigned long long> hs_sums(n_sums);
    HX_CUDA(cudaMemcpyAsync(hs_sums.data(), h->a_sums.p, sizeof(unsigned long long) * n_sums, cudaMemcpyDeviceToHost, st));
    HX_CUDA(cudaStreamSynchronize(st));
    const SupSums s(hs_sums.data(), H);
    const unsigned long long err = *s.err;
    if (err & SUP_ERR_HAP) {
        hx_set_error("hx_read_classes: haplotype code > 6 at a site in 1..N");
        return HX_E_ARG;
    }
    if (err) {
        hx_set_error("hx_read_classes: invalid packed read(s): %s%s",
                     (err & SUP_ERR_RANGE) ? "[read leaves [1,N]] " : "", (err & SUP_ERR_CODE) ? "[allele code > 6]" : "");
        return HX_E_READ;
    }
    for (int i = 0; i < H; ++i)                                  // the singleton classes {h}
        if (s.unique[i]) merged[std::vector<int32_t>{i}] += (int64_t)s.unique[i];
    hx_classes *cl = new (std::nothrow) hx_classes;
    if (!cl) return HX_E_NOMEM;
    cl->off.reserve(merged.size() + 1);
    cl->count.reserve(merged.size());
    cl->off.push_back(0);
    for (const auto &kv : merged) {
        cl->members.insert(cl->members.end(), kv.first.begin(), kv.first.end());
        cl->off.push_back((int64_t)cl->members.size());
        cl->count.push_back(kv.second);
    }
    h->a_cls = cl;
    for (int i = 0; i < 3; ++i) totals[i] = (int64_t)s.totals[i];
    *n_classes = (int64_t)cl->count.size();
    *n_members = (int64_t)cl->members.size();
    return HX_OK;
}

extern "C" int hx_read_classes_get(hx_matrix *h, int64_t *class_off, int32_t *members, int64_t *count) {
    HX_CHECK_ARG(h && class_off && count);
    if (!h->a_cls) {
        hx_set_error("hx_read_classes_get: no classes (hx_read_classes has not succeeded on this handle)");
        return HX_E_STATE;
    }
    const hx_classes &cl = *h->a_cls;
    HX_CHECK_ARG(members || cl.members.empty());
    std::copy(cl.off.begin(), cl.off.end(), class_off);
    std::copy(cl.members.begin(), cl.members.end(), members);
    std::copy(cl.count.begin(), cl.count.end(), count);
    return HX_OK;
}

// The CSR checks of hx_em_abundance and hx_em_bootstrap (HX_E_ARG), and T = the sum of the counts.
int hx_check_classes(int32_t n_haps, int64_t n_classes, const int64_t *class_off, const int32_t *members,
                     const int64_t *count, int64_t *total) {
    const int H = n_haps;
    int64_t T = 0;
    if (n_classes) HX_CHECK_ARG(class_off[0] == 0);
    for (int64_t c = 0; c < n_classes; ++c) {
        const int64_t a = class_off[c], b = class_off[c + 1];
        HX_CHECK_ARG(b > a);                                     // a class has members
        HX_CHECK_ARG(count[c] >= 1);
        for (int64_t j = a; j < b; ++j) {
            HX_CHECK_ARG(members[j] >= 0 && members[j] < H);
            HX_CHECK_ARG(j == a || members[j] > members[j - 1]);
        }
        if (c > 0)
            HX_CHECK_ARG(std::lexicographical_compare(members + class_off[c - 1], members + a, members + a, members + b));
        T += count[c];
    }
    *total = T;
    return HX_OK;
}

// The EM of DESIGN.md §4 K7, in exactly its operation order, so that oracle/abundance_oracle.py reproduces it bit for
// bit.  Host code: the classes are few.  No step may be contracted to an FMA: the x86-64 baseline the library is
// built for has none, and build.py passes no -march that would add it.
extern "C" int hx_em_abundance(int32_t n_haps, int64_t n_classes, const int64_t *class_off, const int32_t *members,
                               const int64_t *count, int32_t max_iter, double tol, double *pi, int32_t *n_iter,
                               int32_t *converged, double *loglik) {
    HX_CHECK_ARG(n_haps >= 1 && n_classes >= 0 && max_iter >= 0 && tol >= 0.0 && pi && n_iter && converged && loglik);
    HX_CHECK_ARG(n_classes == 0 || (class_off && members && count));
    const int H = n_haps;
    int64_t T = 0;
    if (const int rc = hx_check_classes(H, n_classes, class_off, members, count, &T)) return rc;
    if (T == 0) {
        for (int h = 0; h < H; ++h) pi[h] = 0.0;
        *n_iter = 0;
        *converged = 1;
        *loglik = 0.0;
        return HX_OK;
    }
    std::vector<double> acc(H);
    for (int h = 0; h < H; ++h) pi[h] = 1.0 / H;
    double delta = INFINITY;
    int32_t it = 0;
    while (it < max_iter) {
        ++it;
        std::fill(acc.begin(), acc.end(), 0.0);
        for (int64_t c = 0; c < n_classes; ++c) {
            double z = 0.0;
            for (int64_t j = class_off[c]; j < class_off[c + 1]; ++j) z += pi[members[j]];
            for (int64_t j = class_off[c]; j < class_off[c + 1]; ++j) acc[members[j]] += (double)count[c] * (pi[members[j]] / z);
        }
        delta = 0.0;
        for (int h = 0; h < H; ++h) {
            const double nw = acc[h] / (double)T;
            delta = std::max(delta, fabs(nw - pi[h]));
            pi[h] = nw;
        }
        if (delta <= tol) break;
    }
    double ll = 0.0;
    for (int64_t c = 0; c < n_classes; ++c) {
        double z = 0.0;
        for (int64_t j = class_off[c]; j < class_off[c + 1]; ++j) z += pi[members[j]];
        ll += (double)count[c] * log10(z);
    }
    *n_iter = it;
    *converged = delta <= tol;
    *loglik = ll;
    return HX_OK;
}
