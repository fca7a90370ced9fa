// K1, long reads (k up to thousands of SNPs per read: ONT-like, BASELINE configs[3]).
//
// Same pair-expansion semantics as ingest.cu (gretel/util.py:226-286), organised as
// owner-computes so that no atomics are needed for the O(k^2) bulk:
//
//   k_lr_frames     per group of 32 consecutive (rank-sorted) reads: the site range it covers
//   k_scan_*        exclusive scans (plane offsets, running max of the group ends)
//   k_lr_transpose  warp per group: warp ballots turn the 32 reads into per-site bit-planes
//                   (A,C,G,T,N,- masks, 32 B per site) in global memory; sentinels, totals and
//                   the (never seen in BAM data) '_' allele are handled here per read
//   k_lr_site_index per site: first group that reaches it / first group that starts after it
//   k_lr_tiles      CTA per 16x32 tile of site pairs (pi,pj); each thread owns one band cell,
//                   loops over the groups that cover the tile, counts 32 reads with 30 x
//                   (AND, POPC, ADD) in registers and adds its cell to the band once with plain
//                   stores: every band cell has exactly one writer.
#include <limits.h>

#include "hx_internal.cuh"
#include "ingest_common.cuh"
#include "scan.cuh"

namespace {

constexpr int LR_TI = 16, LR_TJ = 32;

// ---- group frames ------------------------------------------------------------------------
__global__ void k_lr_frames(const int32_t *__restrict__ rank, const int64_t *__restrict__ off, int64_t n_reads,
                            int N, int W, int32_t *__restrict__ g_lo, int64_t *__restrict__ g_len,
                            int32_t *__restrict__ g_hi, int *__restrict__ err) {
    const int lane = threadIdx.x & 31;
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_groups = (n_reads + 31) >> 5;
    if (g >= n_groups) return;
    const int64_t idx = g * 32 + lane;
    int lo = INT_MAX, hi = 0;
    if (idx < n_reads) {
        const int64_t k = off[idx + 1] - off[idx];
        const int r = rank[idx];
        if (k >= 2) {
            if (!read_fits(r, k, N, W)) atomicOr(err, 1);
            else { lo = r; hi = r + (int)k; }
        }
    }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    if (lane == 0) {
        const bool any = hi > 0;
        g_lo[g] = any ? lo : (g ? INT_MIN : 0);   // patched below: empty groups inherit order from neighbours
        g_len[g] = any ? (int64_t)(hi - lo) : 0;
        g_hi[g] = any ? hi : 0;
    }
}

// empty groups (no read with >= 2 SNPs) must not break the monotone search keys
__global__ void k_lr_fix_empty(int32_t *__restrict__ g_lo, const int64_t *__restrict__ g_len, int64_t n_groups,
                               const int32_t *__restrict__ rank, int64_t n_reads) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    if (g_len[g] == 0) g_lo[g] = rank[min(g * 32, n_reads - 1)] < 0 ? 0 : rank[min(g * 32, n_reads - 1)];
}

// ---- transpose -----------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_lr_transpose(const int32_t *__restrict__ rank, const int64_t *__restrict__ off,
               const uint8_t *__restrict__ codes, int64_t n_reads, int N, int W,
               const int32_t *__restrict__ g_lo, const int64_t *__restrict__ g_len,
               const int64_t *__restrict__ g_off, uint4 *__restrict__ planes, const HxCnt cnt,
               unsigned long long *__restrict__ totals, int *__restrict__ err,
               const int *__restrict__ sorted_flag) {
    if (!*sorted_flag) return;                       // the generic fallback launch takes over
    const int lane = threadIdx.x & 31;
    const int64_t n_groups = (n_reads + 31) >> 5;
    const int64_t gstride = ((int64_t)gridDim.x * blockDim.x) >> 5;
    unsigned long long t_slices = 0, t_cov = 0, t_sent = 0, t_crumbs = 0;
    for (int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < n_groups; g += gstride) {
        const int64_t idx = g * 32 + lane;
        int64_t o = 0;
        int k = 0, r = 0;
        if (idx < n_reads) {
            o = off[idx];
            const int64_t k64 = off[idx + 1] - o;
            r = rank[idx];
            if (k64 >= 2 && read_fits(r, k64, N, W)) k = (int)k64;
        }
        t_slices += k >= 2;
        const int lo = g_lo[g];
        const int len = (int)g_len[g];
        uint4 *out = planes + 2 * g_off[g];
        const uint8_t *__restrict__ c = codes + o;
        const int shift = r - lo;                         // site t of the frame is position t-shift of the read
        bool has_gap = false;
        for (int t = 0; t < len; ++t) {
            const int u = t - shift;
            unsigned a = 255;
            if (k && u >= 0 && u < k) {
                a = c[u];
                if (a > 6) { atomicOr(err, 2); a = 255; }
            }
            const unsigned mA = __ballot_sync(0xffffffffu, a == 0);
            const unsigned mC = __ballot_sync(0xffffffffu, a == 1);
            const unsigned mG = __ballot_sync(0xffffffffu, a == 2);
            const unsigned mT = __ballot_sync(0xffffffffu, a == 3);
            const unsigned mN = __ballot_sync(0xffffffffu, a == 4);
            const unsigned mD = __ballot_sync(0xffffffffu, a == 5);
            if (lane == 0) {
                out[2 * t] = make_uint4(mA, mC, mG, mT);
                out[2 * t + 1] = make_uint4(mN, mD, 0u, 0u);
            }
            t_cov += (a < 4 || a == 5);
            has_gap |= (a == 6);
        }
        if (k >= 2) add_sentinels(c, c[0], r, k, N, W, cnt, t_sent);
        // '_' as the second allele of a pair is counted (util.py:258 only rejects it as the first);
        // it has no bit-plane: the warp walks such reads position by position
        unsigned gm = __ballot_sync(0xffffffffu, has_gap);
        while (gm) {
            const int src = __ffs(gm) - 1;
            gm &= gm - 1;
            const int64_t o2 = __shfl_sync(0xffffffffu, o, src);
            const int k2 = __shfl_sync(0xffffffffu, k, src);
            const int r2 = __shfl_sync(0xffffffffu, r, src);
            const uint8_t *c2 = codes + o2;
            for (int j = 1; j < k2; ++j) {
                if (c2[j] != HX_SYM_GAP) continue;          // uniform: every lane reads the same byte
                for (int i = lane; i < j; i += 32) {
                    const unsigned a = c2[i];
                    if (sym_valid_from(a)) {
                        atomicAdd(cnt.cell(W, r2 + i + 1, r2 + j + 1) + a * HX_NSYM + HX_SYM_GAP, 1u);
                        t_crumbs++;
                    }
                }
            }
        }
    }
    flush_totals(t_slices, t_crumbs, t_cov, t_sent, totals);
}

// per site s: first group whose running-max end exceeds s (some read so far reaches s), and the
// first group that starts after s
__global__ void k_lr_site_index(const int32_t *__restrict__ g_lo, const int32_t *__restrict__ g_hipm,
                                int64_t n_groups, int N, int64_t *__restrict__ first_reach,
                                int64_t *__restrict__ first_after) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= N) return;
    int64_t a = 0, b = n_groups;
    while (a < b) { const int64_t m = (a + b) >> 1; if (g_hipm[m] > s) b = m; else a = m + 1; }
    first_reach[s] = a;
    a = 0; b = n_groups;
    while (a < b) { const int64_t m = (a + b) >> 1; if (g_lo[m] > s) b = m; else a = m + 1; }
    first_after[s] = a;
}

// ---- tiles ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(LR_TI * LR_TJ, 2)
k_lr_tiles(const uint4 *__restrict__ planes, const int64_t *__restrict__ g_off,
           const int32_t *__restrict__ g_lo, const int64_t *__restrict__ g_len,
           const int64_t *__restrict__ first_reach, const int64_t *__restrict__ first_after, int N, int W,
           int njb, const HxCnt cnt, unsigned long long *__restrict__ totals,
           const int *__restrict__ sorted_flag) {
    if (!*sorted_flag) return;
    const int ib = blockIdx.x / njb, jb = blockIdx.x % njb;
    const int I0 = ib * LR_TI, J0 = I0 + jb * LR_TJ;
    if (J0 >= N) return;
    const int ti = threadIdx.x / LR_TJ, tj = threadIdx.x % LR_TJ;
    const int pi = I0 + ti, pj = J0 + tj;
    const bool valid = pi < N && pj < N && pj > pi && pj - pi <= W;
    // groups that can cover a pair of this tile: started at or before the last pi, reach past J0
    const int ilast = min(I0 + LR_TI - 1, N - 1);
    const int64_t g_begin = first_reach[J0];
    const int64_t g_end = first_after[ilast];
    uint32_t acc[5][6];
#pragma unroll
    for (int a = 0; a < 5; ++a)
#pragma unroll
        for (int b = 0; b < 6; ++b) acc[a][b] = 0;
    for (int64_t g = g_begin; g < g_end; ++g) {
        const int lo = g_lo[g];
        const int len = (int)g_len[g];
        if (lo + len <= J0) continue;                      // uniform: the group ends before the tile's columns
        const int u1 = pi - lo, u2 = pj - lo;
        if (valid && u1 >= 0 && u2 < len) {
            const uint4 *p = planes + 2 * g_off[g];
            const uint4 m1a = __ldg(p + 2 * u1), m1b = __ldg(p + 2 * u1 + 1);
            const uint4 m2a = __ldg(p + 2 * u2), m2b = __ldg(p + 2 * u2 + 1);
            const unsigned x1[5] = {m1a.x, m1a.y, m1a.z, m1a.w, m1b.y};            // A C G T -   (first allele)
            const unsigned x2[6] = {m2a.x, m2a.y, m2a.z, m2a.w, m2b.x, m2b.y};     // A C G T N - (second allele)
#pragma unroll
            for (int a = 0; a < 5; ++a)
#pragma unroll
                for (int b = 0; b < 6; ++b) acc[a][b] += __popc(x1[a] & x2[b]);
        }
    }
    unsigned long long crumbs = 0;
    if (valid) {
        uint32_t *__restrict__ cell = cnt.cell(W, pi + 1, pj + 1);
        const bool shared_cell = cnt.world > 1;                // fused exchange: other GPUs add into it too
#pragma unroll
        for (int a = 0; a < 5; ++a) {
            const int sa = a < 4 ? a : HX_SYM_DEL;
            if (shared_cell) {
#pragma unroll
                for (int b = 0; b < 6; ++b)
                    if (acc[a][b]) atomicAdd(cell + sa * HX_NSYM + b, acc[a][b]);
            } else {
                // single owner: no atomic needed; the six loads of a row go out together, then the stores
                uint32_t old[6];
#pragma unroll
                for (int b = 0; b < 6; ++b) old[b] = cell[sa * HX_NSYM + b];
#pragma unroll
                for (int b = 0; b < 6; ++b)
                    if (acc[a][b]) cell[sa * HX_NSYM + b] = old[b] + acc[a][b];
            }
#pragma unroll
            for (int b = 0; b < 6; ++b) crumbs += acc[a][b];
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) crumbs += __shfl_xor_sync(0xffffffffu, crumbs, o);
    if ((threadIdx.x & 31) == 0 && crumbs) atomicAdd(&totals[1], crumbs);
}

// ---- tiles, planes staged through shared memory (dense coverage) --------------------------------
__global__ void __launch_bounds__(LR_TI * LR_TJ, 2)
k_lr_tiles_staged(const uint4 *__restrict__ planes, const int64_t *__restrict__ g_off,
           const int32_t *__restrict__ g_lo, const int64_t *__restrict__ g_len,
           const int64_t *__restrict__ first_reach, const int64_t *__restrict__ first_after, int N, int W,
           int njb, const HxCnt cnt, unsigned long long *__restrict__ totals,
           const int *__restrict__ sorted_flag) {
    if (!*sorted_flag) return;
    const int ib = blockIdx.x / njb, jb = blockIdx.x % njb;
    const int I0 = ib * LR_TI, J0 = I0 + jb * LR_TJ;
    if (J0 >= N) return;
    const int ti = threadIdx.x / LR_TJ, tj = threadIdx.x % LR_TJ;
    const int pi = I0 + ti, pj = J0 + tj;
    const bool valid = pi < N && pj < N && pj > pi && pj - pi <= W;
    // groups that can cover a pair of this tile: started at or before the last pi, reach past J0
    const int ilast = min(I0 + LR_TI - 1, N - 1);
    const int64_t g_begin = first_reach[J0];
    const int64_t g_end = first_after[ilast];
    uint32_t acc[5][6];
#pragma unroll
    for (int a = 0; a < 5; ++a)
#pragma unroll
        for (int b = 0; b < 6; ++b) acc[a][b] = 0;
    // The planes of the tile's 16 + 32 sites are staged through shared memory with cp.async, two groups
    // ahead of the one being counted (4 stages, one barrier per group): the loads of a group no longer
    // stall the 30 x (AND, POPC, ADD) of the previous ones.
    constexpr int NST = 4, DEPTH = 2, ENT = LR_TI + LR_TJ;
    __shared__ uint4 st_planes[NST][ENT][2];
    __shared__ int st_active[NST];
    const uint32_t st_base = (uint32_t)__cvta_generic_to_shared(&st_planes[0][0][0]);
    for (int64_t g = g_begin; g < g_end + DEPTH; ++g) {
        const int stage = (int)((g - g_begin) % NST);
        if (g < g_end) {
            const int lo = g_lo[g];
            const int len = (int)g_len[g];
            const bool active = lo + len > J0;             // uniform: does the group reach the tile's columns
            if (threadIdx.x == 0) st_active[stage] = active;
            if (active && threadIdx.x < 2 * ENT) {
                const int e = threadIdx.x >> 1, half = threadIdx.x & 1;
                const int site = e < LR_TI ? I0 + e : J0 + (e - LR_TI);
                const int u = site - lo;
                const uint32_t dst = st_base + (uint32_t)(((stage * ENT + e) * 2 + half) * 16);
                if (u >= 0 && u < len) {
                    const uint4 *src = planes + 2 * (g_off[g] + u) + half;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
                } else {
                    asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(dst), "r"(0u) : "memory");
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        const int64_t gc = g - DEPTH;
        if (gc >= g_begin) {
            asm volatile("cp.async.wait_group %0;" ::"n"(DEPTH) : "memory");
            __syncthreads();
            const int sc = (int)((gc - g_begin) % NST);
            if (st_active[sc] && valid) {
                const uint4 m1a = st_planes[sc][ti][0], m1b = st_planes[sc][ti][1];
                const uint4 m2a = st_planes[sc][LR_TI + tj][0], m2b = st_planes[sc][LR_TI + tj][1];
                const unsigned x1[5] = {m1a.x, m1a.y, m1a.z, m1a.w, m1b.y};            // A C G T -   (first allele)
                const unsigned x2[6] = {m2a.x, m2a.y, m2a.z, m2a.w, m2b.x, m2b.y};     // A C G T N - (second allele)
#pragma unroll
                for (int a = 0; a < 5; ++a)
#pragma unroll
                    for (int b = 0; b < 6; ++b) acc[a][b] += __popc(x1[a] & x2[b]);
            }
        }
    }
    unsigned long long crumbs = 0;
    if (valid) {
        uint32_t *__restrict__ cell = cnt.cell(W, pi + 1, pj + 1);
        const bool shared_cell = cnt.world > 1;                // fused exchange: other GPUs add into it too
#pragma unroll
        for (int a = 0; a < 5; ++a) {
            const int sa = a < 4 ? a : HX_SYM_DEL;
            if (shared_cell) {
#pragma unroll
                for (int b = 0; b < 6; ++b)
                    if (acc[a][b]) atomicAdd(cell + sa * HX_NSYM + b, acc[a][b]);
            } else {
                // single owner: no atomic needed; the six loads of a row go out together, then the stores
                uint32_t old[6];
#pragma unroll
                for (int b = 0; b < 6; ++b) old[b] = cell[sa * HX_NSYM + b];
#pragma unroll
                for (int b = 0; b < 6; ++b)
                    if (acc[a][b]) cell[sa * HX_NSYM + b] = old[b] + acc[a][b];
            }
#pragma unroll
            for (int b = 0; b < 6; ++b) crumbs += acc[a][b];
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) crumbs += __shfl_xor_sync(0xffffffffu, crumbs, o);
    if ((threadIdx.x & 31) == 0 && crumbs) atomicAdd(&totals[1], crumbs);
}

}  // namespace

// Scratch owned by the matrix for this path (freed in hx_destroy through hx_lr_free).
struct hx_lr_scratch {
    HxDevBuf<int32_t> g_lo, g_hi, g_hipm;
    HxDevBuf<int64_t> g_len, g_off, first_reach, first_after;
    HxDevBuf<int64_t> part64; HxDevBuf<int32_t> part32; HxDevBuf<int64_t> d_total;
    HxDevBuf<uint4> planes;
};

void hx_lr_free(hx_matrix *h) {
    hx_lr_scratch *s = (hx_lr_scratch *)h->lr_scratch;
    if (!s) return;
    cudaStream_t st = h->stream;
    s->g_lo.release(st); s->g_hi.release(st); s->g_hipm.release(st); s->g_len.release(st); s->g_off.release(st);
    s->first_reach.release(st); s->first_after.release(st);
    s->part64.release(st); s->part32.release(st); s->d_total.release(st); s->planes.release(st);
    delete s;
    h->lr_scratch = nullptr;
}

int hx_launch_ingest_long(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off,
                          const uint8_t *d_codes, int64_t n_reads, const int *sorted_flag) {
    if (!h->lr_scratch) h->lr_scratch = new hx_lr_scratch();
    hx_lr_scratch *s = (hx_lr_scratch *)h->lr_scratch;
    cudaStream_t st = h->stream;
    const int N = h->N, W = h->W;
    const int64_t ng = (n_reads + 31) >> 5;
    constexpr int ITEMS = 16;
    const int64_t nblk = (ng + 256 * ITEMS - 1) / (256 * ITEMS);
    HX_CUDA(s->g_lo.grow(sizeof(int32_t) * ng, st));
    HX_CUDA(s->g_hi.grow(sizeof(int32_t) * ng, st));
    HX_CUDA(s->g_hipm.grow(sizeof(int32_t) * ng, st));
    HX_CUDA(s->g_len.grow(sizeof(int64_t) * ng, st));
    HX_CUDA(s->g_off.grow(sizeof(int64_t) * ng, st));
    HX_CUDA(s->first_reach.grow(sizeof(int64_t) * ((int64_t)N + 1), st));
    HX_CUDA(s->first_after.grow(sizeof(int64_t) * ((int64_t)N + 1), st));
    HX_CUDA(s->part64.grow(sizeof(int64_t) * nblk, st));
    HX_CUDA(s->part32.grow(sizeof(int32_t) * nblk, st));
    HX_CUDA(s->d_total.grow(sizeof(int64_t), st));

    k_lr_frames<<<(unsigned)((ng * 32 + 255) / 256), 256, 0, st>>>(d_rank, d_off, n_reads, N, W, s->g_lo.p, s->g_len.p,
                                                                   s->g_hi.p, h->d_err.p);
    k_lr_fix_empty<<<(unsigned)((ng + 255) / 256), 256, 0, st>>>(s->g_lo.p, s->g_len.p, ng, d_rank, n_reads);
    // plane offsets = exclusive sum of the frame lengths; running max of the group ends
    k_scan_partials<int64_t, 0, ITEMS><<<(unsigned)nblk, 256, 0, st>>>(s->g_len.p, ng, s->part64.p);
    k_scan_spine<int64_t, 0><<<1, 32, 0, st>>>(s->part64.p, nblk, s->d_total.p);
    k_scan_apply<int64_t, 0, ITEMS, true><<<(unsigned)nblk, 256, 0, st>>>(s->g_len.p, ng, s->part64.p, s->g_off.p);
    k_scan_partials<int32_t, 1, ITEMS><<<(unsigned)nblk, 256, 0, st>>>(s->g_hi.p, ng, s->part32.p);
    k_scan_spine<int32_t, 1><<<1, 32, 0, st>>>(s->part32.p, nblk, nullptr);
    k_scan_apply<int32_t, 1, ITEMS, false><<<(unsigned)nblk, 256, 0, st>>>(s->g_hi.p, ng, s->part32.p, s->g_hipm.p);
    h->use.launches += 8;
    HX_CUDA(cudaGetLastError());
    // The plane buffer is sized by a bound instead of the scan total (no device->host round trip, so chunks of long
    // reads can overlap their copies like the short ones): a group's frame spans the ranks of its 32 rank-sorted
    // reads plus one read, and the rank ranges of consecutive groups do not overlap.
    const int64_t total_sites_bound = (int64_t)N + 1 + ng * ((int64_t)W + 1);
    HX_CUDA(s->planes.grow(sizeof(uint4) * (2 * total_sites_bound + 2), st));

    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    const int64_t want = (ng * 32 + 255) / 256;
    const int tgrid = (int)(want < (int64_t)sms * 8 ? want : (int64_t)sms * 8);
    k_lr_transpose<<<tgrid, 256, 0, st>>>(d_rank, d_off, d_codes, n_reads, N, W, s->g_lo.p, s->g_len.p, s->g_off.p,
                                          s->planes.p, hx_cnt_ref(h), h->d_totals.p, h->d_err.p, sorted_flag);
    k_lr_site_index<<<(N + 255) / 256, 256, 0, st>>>(s->g_lo.p, s->g_hipm.p, ng, N, s->first_reach.p, s->first_after.p);
    const int nib = (N + LR_TI - 1) / LR_TI;
    const int njb = (W + LR_TI - 1) / LR_TJ + 1;            // J0 = I0 + jb*TJ must reach pi + W for the last row
    // measured (B200, ONT-like reads): with ~10 reads per SNP rank the cp.async-staged tiles win (9.2 vs
    // 11.3 ms for 100k reads), with ~2 per rank the per-group barrier costs more than it hides (3.8 vs 1.4 ms)
    if (n_reads >= 6 * (int64_t)N)
        k_lr_tiles_staged<<<(unsigned)((int64_t)nib * njb), LR_TI * LR_TJ, 0, st>>>(
            s->planes.p, s->g_off.p, s->g_lo.p, s->g_len.p, s->first_reach.p, s->first_after.p, N, W, njb, hx_cnt_ref(h),
            h->d_totals.p, sorted_flag);
    else
        k_lr_tiles<<<(unsigned)((int64_t)nib * njb), LR_TI * LR_TJ, 0, st>>>(
            s->planes.p, s->g_off.p, s->g_lo.p, s->g_len.p, s->first_reach.p, s->first_after.p, N, W, njb, hx_cnt_ref(h),
            h->d_totals.p, sorted_flag);
    h->use.launches += 3;
    HX_CUDA(cudaGetLastError());
    return HX_OK;
}
