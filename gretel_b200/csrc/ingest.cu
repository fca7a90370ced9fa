// K1: pair-expansion ingestion of packed reads into the banded Hansel counts.
// Replaces gretel/util.py:226-286 (+ Hansel.add_observation) of the reference.
//
// Two kernels (chosen per launch, see hx_launch_ingest):
//
//   k1_pairs_red   generic: one warp per read, lanes over the linearised (i,j) triangle,
//                  one fire-and-forget integer reduction (RED) per pair into the band.
//                  Any read order, any k.  Bound by the chip-wide RED rate
//                  (measured 187 G/s on B200, tools/microbench.cu).
//
//   k1_bitsliced   rank-sorted reads with at most BS_KMAX SNPs.  Reads that share a rank
//                  (same first SNP) cover the same site pairs, so 32 of them are
//                  transposed with warp ballots into per-site allele bit-planes
//                  (A,C,G,T masks over the 32 reads); a site pair (t1,t2) then costs
//                  16 x (AND, POPC, ADD) for 32 reads instead of 32 atomics, accumulated
//                  in registers by the thread that owns the pair (warp-aggregation by
//                  construction).  Per-CTA the counts are privatised in a sliding
//                  shared-memory tile (ring of band rows); a row is flushed to HBM with
//                  REDs once no later read of the CTA can touch it.  Rare alleles
//                  (N, -, _), sentinels and totals are handled per read on the side.
#include <atomic>

#include "hx_internal.cuh"
#include "ingest_common.cuh"

namespace {

constexpr int BS_KMAX = 52;      // widest read (in SNPs) the bit-sliced kernel takes
constexpr int BS_GB = 32;        // most groups (of 32 reads) per build/accumulate batch

// The per-pair rules of util.py:254-281 for one (i,j) of one read (sentinels included).
__device__ __forceinline__ void add_pair(const HxCnt cnt, int N, int64_t W, int rk, int i,
                                         int j, unsigned a, unsigned b, unsigned long long &sent) {
    const int pi = rk + i + 1, pj = rk + j + 1;
    atomicAdd(cnt.cell(W, pi, pj) + a * HX_NSYM + b, 1u);            // :267,274,280
    if (i == 0 && j == 1 && rk == 0) {                                          // :262-266
        atomicAdd(cnt.cell(W, 0, 1) + HX_SYM_GAP * HX_NSYM + a, 1u);
        sent++;
    } else if (pj == N && j - i == 1) {                                         // :271-275
        atomicAdd(cnt.cell(W, N, N + 1) + b * HX_NSYM + HX_SYM_GAP, 1u);
        sent++;
    }
}

// One whole read, cooperatively by the calling warp (all 32 lanes converged).
__device__ __forceinline__ void warp_read_generic(const uint8_t *__restrict__ c, int k, int rk, int N,
                                                  int64_t W, const HxCnt cnt,
                                                  unsigned long long &t_crumbs, unsigned long long &t_cov,
                                                  unsigned long long &t_sent, int *err) {
    const int lane = threadIdx.x & 31;
    for (int t = lane; t < k; t += 32) {
        const unsigned a = c[t];
        if (a > 6) atomicOr(err, 2);
        const bool v = sym_valid_from(a);
        t_cov += v;                                                             // util.py:239
        t_crumbs += v ? (unsigned)(k - 1 - t) : 0u;                             // pairs with a valid first allele
    }
    const int64_t npairs = (int64_t)k * (k - 1) / 2;
    const int m = 2 * k - 1;
    for (int64_t q = lane; q < npairs; q += 32) {
        // row-major upper triangle: row i starts at i*(m-i)/2
        const float disc = (float)((int64_t)m * m - 8 * q);
        int i = (int)(((float)m - sqrtf(disc)) * 0.5f);
        i = max(0, min(i, k - 2));
        while ((int64_t)(i + 1) * (m - (i + 1)) / 2 <= q) ++i;
        while ((int64_t)i * (m - i) / 2 > q) --i;
        const int j = i + 1 + (int)(q - (int64_t)i * (m - i) / 2);
        const unsigned a = c[i], b = c[j];
        if (!sym_valid_from(a) || b > 6) continue;
        add_pair(cnt, N, W, rk, i, j, a, b, t_sent);
    }
}

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK)
k1_pairs_red(const int32_t *__restrict__ rank, const int64_t *__restrict__ off,
             const uint8_t *__restrict__ codes, int64_t n_reads, int N, int W,
             const HxCnt cnt, unsigned long long *__restrict__ totals,
             int *__restrict__ err, const int *__restrict__ sorted_flag, int run_if_sorted) {
    // sorted_flag: 1 when the reads are rank-sorted.  run_if_sorted = 0 makes this launch the
    // fallback that only runs when the bit-sliced kernel declined the input; 1 = run regardless;
    // 2 = run only if the flag is set (a pre-decoded chunk that passed its consistency check).
    if (run_if_sorted == 0 && *sorted_flag) return;
    if (run_if_sorted == 2 && !*sorted_flag) return;
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    unsigned long long t_slices = 0, t_crumbs = 0, t_cov = 0, t_sent = 0;
    for (int64_t r = (int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5); r < n_reads; r += nwarps) {
        const int64_t o = off[r];
        const int64_t k64 = off[r + 1] - o;
        if (k64 < 2) continue;                                                  // util.py:230
        const int rk = rank[r];
        if (!read_fits(rk, k64, N, W)) {
            if (lane == 0) atomicOr(err, 1);
            continue;
        }
        if (lane == 0) t_slices++;
        warp_read_generic(codes + o, (int)k64, rk, N, W, cnt, t_crumbs, t_cov, t_sent, err);
    }
    flush_totals(t_slices, t_crumbs, t_cov, t_sent, totals);
}

// One launch instead of two fills: the "sorted" flag starts at 1, run_end at -1 (= no reads of that rank).
__global__ void k_prepass_init(int *__restrict__ flag, int64_t *__restrict__ run_end, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *flag = 1;
    if (i < n) run_end[i] = -1;
}

// Pre-pass over the rank array: clears *flag when the reads are not rank-sorted and records
// where the run of reads of each rank ends (exclusive), so the main kernel never searches.
__global__ void k_prepass(const int32_t *__restrict__ rank, int64_t n_reads, int N, int *__restrict__ flag,
                          int64_t *__restrict__ run_end, int *__restrict__ err) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_reads) return;
    const int r = rank[i];
    if (r < 0 || r > N) atomicOr(err, 1);            // the tensor-core kernel walks run_end and never sees this read
    if (i + 1 < n_reads) {
        const int r2 = rank[i + 1];
        if (r > r2) *flag = 0;
        if (r != r2 && r >= 0 && r <= N) run_end[r] = i + 1;
    } else if (r >= 0 && r <= N) {
        run_end[r] = n_reads;
    }
}

// ------------------------------------------------------------------------------------------
// Bit-sliced kernel.
//
// Shared memory (dynamic):
//   tile   [(kmax+1) rows][(kmax-1) cells][16 u32]   ring of band rows; row = pj % (kmax+1),
//          cell = d-1 (d = pj-pi), 16 = (a,b) in ACGT x ACGT.
//   planes [BS_GB groups][kmax sites] uint4           A,C,G,T masks over the group's 32 reads
//   gk     [BS_GB] int                                 widest read of each group
//   rareq  [BS_GB*32] int                              reads of the batch holding N, - or _
//
// Thread p owns site pair (t1,t2), t2-major (p = t2(t2-1)/2 + t1), relative to the rank
// of the current run of reads, so the pairs covered by reads of k SNPs are the prefix
// p < k(k-1)/2 and warps stay converged.
struct BsLayout {
    int kmax, gb;
    __host__ __device__ size_t tile_u4() const { return (size_t)(kmax + 1) * (kmax - 1) * 4; }
    __host__ __device__ size_t bytes() const {
        return tile_u4() * 16 + (size_t)2 * gb * kmax * 16 + 64 * sizeof(int) + (size_t)2 * gb * 32 * sizeof(int);
    }
};

// Transposes one group of 32 reads (lane = read, kb SNPs each, codes at codes+o) into bit-planes in
// shared memory: planes[t] = {v, b0, b1, -} with bit r of v set when read r holds A/C/G/T at site t and
// (b0,b1) the two low code bits of that allele.  No warp votes (they share the quarter-rate XU pipe with
// POPC): every lane packs 10 sites x 3 flags of its own read into one word and a 32x32 bit-matrix
// transpose over the warp (5 shuffle stages on the ALU) turns "flags of my read" into "reads per flag".
// Returns the widest read of the group; rare_or != 0 marks reads holding N, - or _; x0 = first 4 codes.
template <int KW>
__device__ __forceinline__ int bs_build_group(const uint8_t *__restrict__ codes, int64_t o, int kb,
                                              uint32_t pg_addr, uint32_t &rare_or, uint32_t &x0) {
    const int lane = threadIdx.x & 31;
    const int kg = __reduce_max_sync(0xffffffffu, kb);
    const uint8_t *__restrict__ c = codes + o;
    const unsigned mis = (unsigned)(reinterpret_cast<uintptr_t>(c) & 3u);
    const uint32_t *__restrict__ cw = reinterpret_cast<const uint32_t *>(c - mis);
    const int nw = kb ? (int)((mis + kb + 3) >> 2) : 0;
    uint32_t wd[KW + 1];
#pragma unroll
    for (int w = 0; w <= KW; ++w) wd[w] = w < nw ? __ldg(cw + w) : 0u;
    const unsigned sh = 8u * mis;
    const int kb8 = 8 * kb;
    // Four sites per 32-bit operation: g12[w] = the 3-bit flags (v | b0<<1 | b1<<2, 0 for N/-/_ and past the
    // read's end) of sites 4w..4w+3.  Words the group's widest read does not reach are skipped (warp-uniform).
    uint32_t g12[KW];
    rare_or = 0;
    x0 = 0xffffffffu;
#pragma unroll
    for (int w = 0; w < KW; ++w) {
        g12[w] = 0;
        if (w == 0 || 4 * w < kg) {
            const uint32_t xx = __funnelshift_r(wd[w], wd[w + 1], sh);
            const int c8 = min(max(kb8 - 32 * w, 0), 32);         // valid bits of this word
            uint32_t inval;                                       // bytes past the read's end
            asm("shl.b32 %0, %1, %2;" : "=r"(inval) : "r"(0xffffffffu), "r"(c8));   // shl clamps: c8 = 32 -> 0
            rare_or |= xx & 0xfcfcfcfcu & ~inval;
            const uint32_t x = xx | inval;                        // -> 0xff
            if (w == 0) x0 = x;
            const uint32_t u = (x >> 2) & 0x3f3f3f3fu;            // any of bits 2..7 set => not A/C/G/T
            const uint32_t v = (((u + 0x3f3f3f3fu) & 0x40404040u) >> 6) ^ 0x01010101u;   // 1 per valid byte
            const uint32_t f = ((x & 0x03030303u) * 2u + 0x01010101u) & (v * 7u);        // 2a+1 or 0 per byte
            g12[w] = (f & 7u) | ((f >> 5) & 0x38u) | ((f >> 10) & 0x1c0u) | ((f >> 15) & 0xe00u);
        }
    }
    // which (site, flag) this lane will hold after a transpose: flag index = lane
    const int my_tl = lane / 3, my_plane = lane - 3 * my_tl;
#pragma unroll
    for (int t0 = 0; t0 < 4 * KW; t0 += 10) {
        if (t0 >= kg) break;                                      // warp-uniform
        // flags of my read for sites t0..t0+9: 20 sites are five 12-bit groups
        const int c = t0 / 10, wb = 5 * (c >> 1);
        auto G = [&](int i) -> uint32_t { return i < KW ? g12[i] : 0u; };
        uint32_t row = (c & 1) ? ((G(wb + 2) >> 6) | (G(wb + 3) << 6) | (G(wb + 4) << 18))
                               : (G(wb) | (G(wb + 1) << 12) | ((G(wb + 2) & 0x3fu) << 24));
        // 32x32 bit transpose across the warp: afterwards bit r of `row` = flag `lane` of read r.  A stage keeps
        // half of the own word and takes the other half from the partner, shifted by j; as a rotation (the
        // wrapped bits fall outside the mask) that is shuffle + funnel shift + one bit-select.
#pragma unroll
        for (int j = 16; j >= 1; j >>= 1) {
            const uint32_t m = j == 16 ? 0x0000ffffu : j == 8 ? 0x00ff00ffu : j == 4 ? 0x0f0f0f0fu
                             : j == 2 ? 0x33333333u : 0x55555555u;
            const bool up = (lane & j) != 0;
            const uint32_t take = up ? m : ~m;                    // bits that come from the partner
            const uint32_t y = __shfl_xor_sync(0xffffffffu, row, j);
            const uint32_t yr = __funnelshift_l(y, y, up ? 32 - j : j);
            row = (row & ~take) | (yr & take);
        }
        const int t = t0 + my_tl;
        if (lane < 30 && t < kg)
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(pg_addr + (uint32_t)(t * 16 + my_plane * 4)), "r"(row) : "memory");
    }
    return kg;
}

// One thread's site pair (a1,a2) over the nb groups of a plane buffer: 16 x (AND, POPC, ADD) per group
// of 32 reads.  Shared-window byte addresses are kept in registers and advanced per group (the compiler
// otherwise rebuilds them from the kernel parameters in every iteration).
__device__ __forceinline__ void bs_accumulate(uint32_t (&acc)[16], uint32_t buf_saddr, uint32_t gk_addr, int a1, int a2,
                                              int nb, int kmax) {
    uint32_t p1 = buf_saddr + (uint32_t)a1 * 16u, p2 = buf_saddr + (uint32_t)a2 * 16u;
    uint32_t gstep = (uint32_t)kmax * 16u;
    asm volatile("" : "+r"(p1), "+r"(p2), "+r"(gstep), "+r"(gk_addr));
    for (int g = 0; g < nb; ++g, p1 += gstep, p2 += gstep, gk_addr += 4u) {
        int kg;
        asm volatile("ld.shared.s32 %0, [%1];" : "=r"(kg) : "r"(gk_addr));
        if (a2 < kg) {
            uint4 m1, m2;
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(m1.x), "=r"(m1.y), "=r"(m1.z), "=r"(m1.w) : "r"(p1));
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(m2.x), "=r"(m2.y), "=r"(m2.z), "=r"(m2.w) : "r"(p2));
            // planes hold (v, b0, b1): A = v&~b0&~b1, C = b0&~b1, G = b1&~b0, T = b0&b1
            const unsigned x1[4] = {m1.x & ~(m1.y | m1.z), m1.y & ~m1.z, m1.z & ~m1.y, m1.y & m1.z};
            const unsigned x2[4] = {m2.x & ~(m2.y | m2.z), m2.y & ~m2.z, m2.z & ~m2.y, m2.y & m2.z};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) acc[a * 4 + b] += __popc(x1[a] & x2[b]);
        }
    }
}

// One batch of up to `gb` groups (32 reads each) out of a run of reads that share rank r.
struct BsBatch {
    int64_t start;      // first read
    int n;              // reads in the batch (0 = no batch)
    int r;              // rank of the run
    bool first, last;   // first / last batch of its run (within this CTA's slice)
};

template <int KW, int NP, int MAXT, int MINB, bool FUSED>
__global__ void __launch_bounds__(MAXT, MINB)
k1_bitsliced(const int32_t *__restrict__ rank, const int64_t *__restrict__ off,
             const uint8_t *__restrict__ codes, int64_t n_reads, int N, int W, int kmax, int gb,
             const HxCnt cnt_in, unsigned long long *__restrict__ totals,
             int *__restrict__ err, const int *__restrict__ sorted_flag,
             const int64_t *__restrict__ run_end) {
    extern __shared__ uint4 smem4[];
    const HxCnt cnt = cnt_in.for_build<FUSED>();
    if (!*sorted_flag) return;                       // the generic fallback launch takes over
    const int rows = kmax + 1, cells = kmax - 1;
    uint4 *const tile = smem4;
    uint32_t *const tile32 = reinterpret_cast<uint32_t *>(tile);
    uint4 *const planes0 = tile + (size_t)rows * cells * 4;          // two buffers of gb*kmax uint4
    int *const gk0 = reinterpret_cast<int *>(planes0 + (size_t)2 * gb * kmax);   // two buffers of 32 ints
    int *const rareq0 = gk0 + 64;                                     // two buffers of gb*32 ints
    const uint32_t planes_saddr = (uint32_t)__cvta_generic_to_shared(planes0);
    const uint32_t gk_saddr = (uint32_t)__cvta_generic_to_shared(gk0);
    __shared__ int s_rare_n[3];                      // rotating: built / consumed / being cleared
    __shared__ int s_claim[3];                       // next group to transpose (same rotation): warps claim work

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    int64_t lo, hi;                                  // equal shares of the work, not of the read count
    hx_weighted_slice(rank, off, n_reads, HX_SLICE_READ_W, HX_SLICE_RANK_W, lo, hi);
    if (lo >= hi) return;

    for (size_t w = threadIdx.x; w < (size_t)rows * cells * 4; w += blockDim.x) tile[w] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) { s_rare_n[0] = s_rare_n[1] = s_rare_n[2] = 0; s_claim[0] = s_claim[1] = s_claim[2] = 0; }
    const uint32_t pf_bytes = (uint32_t)gb * 32u * (uint32_t)(kmax > 40 ? 32 : 18);   // ~ one batch of codes
    int rc_build = 1, rc_cons = 0, rc_clear = 2;      // indices into s_rare_n, rotated every phase

    // this thread's site pair(s)
    int t1[NP], t2[NP];
#pragma unroll
    for (int q = 0; q < NP; ++q) {
        const int p = threadIdx.x + q * blockDim.x;
        int b = (int)((1.0f + sqrtf(1.0f + 8.0f * (float)p)) * 0.5f);
        while (b * (b - 1) / 2 > p) --b;
        while ((b + 1) * b / 2 <= p) ++b;
        t2[q] = b;
        t1[q] = p - b * (b - 1) / 2;
    }
    unsigned long long t_crumbs = 0;
    unsigned n_slices = 0, n_codes = 0, n_notcov = 0, n_sent = 0, n_rcrumbs = 0, errbits = 0;
    int64_t flushed_upto = (int64_t)rank[lo] + 1;    // rows pj <= flushed_upto hold nothing
    uint32_t acc[NP][16];
    int run_kmax = 0, rbase = 0;

    // batch scheduler state (identical in every thread)
    int64_t cur = lo, run_hi = lo;
    int run_r = 0;
    BsBatch prev{0, 0, 0, false, false};
    int buf = 0;
    int prev_aw = 0;                                 // warps that own active pairs in `prev`
    __syncthreads();

    for (;;) {
        // ---- next batch -----------------------------------------------------------------------
        BsBatch next{0, 0, 0, false, false};
        if (cur < hi) {
            next.first = cur >= run_hi;
            if (next.first) {
                run_r = rank[cur];
                run_hi = cur + 1;
                if (run_r >= 0 && run_r <= N) {      // ranks the pre-pass indexed
                    run_hi = run_end[run_r];
                    if (run_hi > hi) run_hi = hi;
                }
            }
            next.start = cur;
            next.r = run_r;
            next.n = (int)min((int64_t)gb * 32, run_hi - cur);
            cur += next.n;
            next.last = cur >= run_hi;
            if (threadIdx.x == 0 && cur < hi) {          // the batch after `next`: its offsets and first rank
                const int64_t ahead = min((int64_t)gb * 32 + 1, hi - cur + 1);
                bs_prefetch_l2(off + cur, (uint32_t)(ahead * 8));
                bs_prefetch_l2(rank + cur, 16);
            }
        }
        if (!prev.n && !next.n) break;

        // ---- consume `prev` (planes buffer buf^1) ---------------------------------------------
        if (prev.n) {
            const int pb = buf ^ 1;
            const int *gk = gk0 + pb * 32;
            const int nb = (prev.n + 31) >> 5;
            const int r = prev.r;
            if (prev.first) {
                // rows pj <= r+1 can no longer be touched by this CTA (reads of rank >= r start at pj = r+2)
                if ((int64_t)r + 1 > flushed_upto) {
                    const int64_t last = min((int64_t)r + 1, flushed_upto + rows - 2);
                    t_crumbs += bs_flush_rows(tile32, rows, cells, flushed_upto + 1, last, W, cnt, blockDim.x, true);
                    flushed_upto = (int64_t)r + 1;
                    __syncthreads();                 // the retired ring slots may be reused by this run's tile add
                }
                rbase = (int)(((int64_t)r + 1) % rows);   // ring row of pj = r+1+t2 is rbase+t2 (mod rows)
                run_kmax = 0;
#pragma unroll
                for (int q = 0; q < NP; ++q)
#pragma unroll
                    for (int x = 0; x < 16; ++x) acc[q][x] = 0;
            }
            const int bkm = __reduce_max_sync(0xffffffffu, lane < nb ? gk[lane] : 0);
            run_kmax = max(run_kmax, bkm);
            prev_aw = (bkm * (bkm - 1) / 2 + 31) >> 5;
#pragma unroll
            for (int q = 0; q < NP; ++q) {
                if (t2[q] < bkm) bs_accumulate(acc[q], planes_saddr + (uint32_t)(pb * gb * kmax) * 16u, gk_saddr + pb * 128u,
                                               t1[q], t2[q], nb, kmax);
            }
            if (prev.last) {
                // add this run's counts into the sliding tile (each cell has one owner thread)
#pragma unroll
                for (int q = 0; q < NP; ++q) {
                    if (t2[q] < run_kmax) {
                        int row = rbase + t2[q];
                        if (row >= rows) row -= rows;
                        const int d = t2[q] - t1[q];
                        uint4 *cell = tile + ((size_t)row * cells + (d - 1)) * 4;
#pragma unroll
                        for (int x = 0; x < 4; ++x) {
                            uint4 v = cell[x];
                            v.x += acc[q][4 * x + 0]; v.y += acc[q][4 * x + 1];
                            v.z += acc[q][4 * x + 2]; v.w += acc[q][4 * x + 3];
                            cell[x] = v;
                        }
                    }
                }
            }
            // reads with rare alleles, one warp per read (warps without active pairs get here first)
            const int nrare = s_rare_n[rc_cons];
            const int *rareq = rareq0 + (size_t)pb * gb * 32;
            for (int qi = nwarps - 1 - warp; qi < nrare; qi += nwarps) {
                const int64_t idx = prev.start + rareq[qi];
                const int64_t o = off[idx];
                const int kb = (int)(off[idx + 1] - o);
                bs_rare_read(codes + o, kb, r, W, cnt, n_rcrumbs, n_notcov, errbits);
            }
        } else {
            prev_aw = 0;
        }

        // ---- produce `next` (planes buffer buf): one warp per group, pair-less warps first -----
        if (next.n) {
            int *gk = gk0 + buf * 32;
            int *rareq = rareq0 + (size_t)buf * gb * 32;
            const int nb = (next.n + 31) >> 5;
            const int r = next.r;
            const int64_t run_stop = next.start + next.n;
            // every warp claims groups until none is left: warps without active pairs of `prev` get here
            // first and do most of the transposing, the pair-owning warps join when they are done
            for (;;) {
                int g = 0;
                if (lane == 0) g = atomicAdd(&s_claim[rc_build], 1);
                g = __shfl_sync(0xffffffffu, g, 0);
                if (g >= nb) break;
                const int64_t idx = next.start + (int64_t)g * 32 + lane;
                int64_t o = 0;
                int kb = 0;
                if (idx < run_stop) {
                    o = off[idx];
                    const int64_t k64 = off[idx + 1] - o;
                    if (k64 >= 2) {
                        if (!read_fits(r, k64, N, W)) errbits |= 1;
                        else kb = (int)k64;
                    }
                    // last read of the batch: the next batch's codes start right behind it
                    if (idx + 1 == run_stop && idx + 1 < hi) bs_prefetch_l2(codes + o + k64, pf_bytes);
                }
                n_slices += kb >= 2;
                n_codes += kb;
                uint32_t rare_or, x0;
                const int kg = bs_build_group<KW>(codes, o, kb, planes_saddr + (uint32_t)((buf * gb + g) * kmax) * 16u,
                                                  rare_or, x0);
                if (lane == 0) gk[g] = kg;
                if (kb >= 2) {
                    add_sentinels(codes + o, x0 & 0xffu, r, kb, N, W, cnt, n_sent);
                    if (rare_or) rareq[atomicAdd(&s_rare_n[rc_build], 1)] = g * 32 + lane;
                }
            }
        }
        if (threadIdx.x == 0) { s_rare_n[rc_clear] = 0; s_claim[rc_clear] = 0; }   // used one phase ago, reused one phase ahead
        __syncthreads();
        prev = next;
        buf ^= 1;
        { const int t = rc_clear; rc_clear = rc_cons; rc_cons = rc_build; rc_build = t; }
    }
    __syncthreads();
    t_crumbs += bs_flush_rows(tile32, rows, cells, flushed_upto + 1, flushed_upto + rows - 1, W, cnt, blockDim.x, true);
    if (errbits) atomicOr(err, (int)errbits);
    // covered SNPs (util.py:239) = all codes of the kept reads minus the N and _ among them
    flush_totals(n_slices, t_crumbs + n_rcrumbs, (unsigned long long)n_codes - n_notcov, n_sent, totals);
}

// ------------------------------------------------------------------------------------------
// Warp-specialised variant of the bit-sliced kernel: dedicated builder warps transpose batches
// into a ring of NBUF plane buffers while the pair-owning warps count; the two sides only meet
// on mbarriers (full[b]: builders -> counters, empty[b]: counters -> builders), so nobody waits
// at a CTA-wide barrier.  The pair warps keep the sliding tile and synchronise among themselves
// with a named barrier at run boundaries.
constexpr int WS_NBUF = 3;

struct WsLayout {
    int kmax, gb;
    __host__ __device__ size_t tile_u4() const { return (size_t)(kmax + 1) * (kmax - 1) * 4; }
    __host__ __device__ size_t bytes() const {
        return tile_u4() * 16 + (size_t)WS_NBUF * gb * kmax * 16 + (size_t)WS_NBUF * 32 * sizeof(int);
    }
};

template <int KW, int NP, int MAXT, int MINB, bool FUSED>
__global__ void __launch_bounds__(MAXT, MINB)
k1_bitsliced_ws(const int32_t *__restrict__ rank, const int64_t *__restrict__ off,
                const uint8_t *__restrict__ codes, int64_t n_reads, int N, int W, int kmax, int gb, int pw,
                const HxCnt cnt_in, unsigned long long *__restrict__ totals,
                int *__restrict__ err, const int *__restrict__ sorted_flag,
                const int64_t *__restrict__ run_end) {
    extern __shared__ uint4 smem4[];
    const HxCnt cnt = cnt_in.for_build<FUSED>();
    __shared__ __align__(8) unsigned long long s_full[WS_NBUF], s_empty[WS_NBUF];
    if (!*sorted_flag) return;                       // the generic fallback launch takes over
    const int rows = kmax + 1, cells = kmax - 1;
    uint4 *const tile = smem4;
    uint32_t *const tile32 = reinterpret_cast<uint32_t *>(tile);
    uint4 *const planes0 = tile + (size_t)rows * cells * 4;                      // WS_NBUF x gb x kmax uint4
    int *const gk0 = reinterpret_cast<int *>(planes0 + (size_t)WS_NBUF * gb * kmax);   // WS_NBUF x 32
    const uint32_t planes_saddr = (uint32_t)__cvta_generic_to_shared(planes0);
    const uint32_t gk_saddr = (uint32_t)__cvta_generic_to_shared(gk0);

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int bw = nwarps - pw;                      // builder warps
    const bool is_pair = warp < pw;
    const int npt = pw * 32;                         // threads that own site pairs
    int64_t lo, hi;                                  // equal shares of the work, not of the read count
    hx_weighted_slice(rank, off, n_reads, HX_SLICE_READ_W, HX_SLICE_RANK_W, lo, hi);
    if (lo >= hi) return;

    for (size_t w = threadIdx.x; w < (size_t)rows * cells * 4; w += blockDim.x) tile[w] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        for (int b = 0; b < WS_NBUF; ++b) {
            hx_mbar_init(hx_smem_u32(&s_full[b]), bw);
            hx_mbar_init(hx_smem_u32(&s_empty[b]), pw);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    unsigned long long t_crumbs = 0;
    unsigned n_slices = 0, n_codes = 0, n_notcov = 0, n_sent = 0, n_rcrumbs = 0, errbits = 0;
    const uint32_t pf_bytes = (uint32_t)gb * 32u * (uint32_t)(kmax > 40 ? 32 : 18);   // ~ one batch of codes

    // batch scheduler (identical in every warp)
    int64_t cur = lo, run_hi = lo;
    int run_r = 0;
    unsigned bi = 0;                                 // batch index

    if (!is_pair) {
        // ================================ builders ==========================================
        const int bwid = warp - pw;
        for (;; ++bi) {
            if (cur >= hi) break;
            if (cur >= run_hi) {
                run_r = rank[cur];
                run_hi = cur + 1;
                if (run_r >= 0 && run_r <= N) {
                    run_hi = run_end[run_r];
                    if (run_hi > hi) run_hi = hi;
                }
            }
            const int64_t bstart = cur;
            const int bn = (int)min((int64_t)gb * 32, run_hi - cur);
            cur += bn;
            if (bwid == 0 && lane == 0 && cur < hi) {      // the next batch: its offsets and first rank
                const int64_t ahead = min((int64_t)gb * 32 + 1, hi - cur + 1);
                bs_prefetch_l2(off + cur, (uint32_t)(ahead * 8));
                bs_prefetch_l2(rank + cur, 16);
            }
            const int r = run_r;
            const int nb = (bn + 31) >> 5;
            const int b = bi % WS_NBUF;
            hx_mbar_wait(hx_smem_u32(&s_empty[b]), ((bi / WS_NBUF) & 1) ^ 1);
            int *gk = gk0 + b * 32;
            const int64_t run_stop = bstart + bn;
            for (int g = bwid; g < nb; g += bw) {
                const int64_t idx = bstart + (int64_t)g * 32 + lane;
                int64_t o = 0;
                int kb = 0;
                if (idx < run_stop) {
                    o = off[idx];
                    const int64_t k64 = off[idx + 1] - o;
                    if (k64 >= 2) {
                        if (!read_fits(r, k64, N, W)) errbits |= 1;
                        else kb = (int)k64;
                    }
                    // last read of the batch: the next batch's codes start right behind it
                    if (idx + 1 == run_stop && idx + 1 < hi) bs_prefetch_l2(codes + o + k64, pf_bytes);
                }
                n_slices += kb >= 2;
                n_codes += kb;
                uint32_t rare_or, x0;
                const int kg = bs_build_group<KW>(codes, o, kb, planes_saddr + (uint32_t)((b * gb + g) * kmax) * 16u,
                                                  rare_or, x0);
                if (lane == 0) gk[g] = kg;
                if (kb >= 2) add_sentinels(codes + o, x0 & 0xffu, r, kb, N, W, cnt, n_sent);
                // reads holding N, - or _: their pairs with such an allele are added right here by the warp
                unsigned rm = __ballot_sync(0xffffffffu, kb >= 2 && rare_or != 0);
                while (rm) {
                    const int src = __ffs(rm) - 1;
                    rm &= rm - 1;
                    const int64_t o2 = __shfl_sync(0xffffffffu, o, src);
                    const int k2 = __shfl_sync(0xffffffffu, kb, src);
                    bs_rare_read(codes + o2, k2, r, W, cnt, n_rcrumbs, n_notcov, errbits);
                }
            }
            __syncwarp();
            if (lane == 0) ws_mbar_arrive(hx_smem_u32(&s_full[b]));
        }
    } else {
        // ================================ pair owners =======================================
        int t1[NP], t2[NP];
#pragma unroll
        for (int q = 0; q < NP; ++q) {
            const int p = threadIdx.x + q * npt;
            int b = (int)((1.0f + sqrtf(1.0f + 8.0f * (float)p)) * 0.5f);
            while (b * (b - 1) / 2 > p) --b;
            while ((b + 1) * b / 2 <= p) ++b;
            t2[q] = b;
            t1[q] = p - b * (b - 1) / 2;
        }
        int64_t flushed_upto = (int64_t)rank[lo] + 1;
        uint32_t acc[NP][16];
        int run_kmax = 0, rbase = 0;
        for (;; ++bi) {
            if (cur >= hi) break;
            const bool first = cur >= run_hi;
            if (first) {
                run_r = rank[cur];
                run_hi = cur + 1;
                if (run_r >= 0 && run_r <= N) {
                    run_hi = run_end[run_r];
                    if (run_hi > hi) run_hi = hi;
                }
            }
            const int bn = (int)min((int64_t)gb * 32, run_hi - cur);
            cur += bn;
            const bool last = cur >= run_hi;
            const int r = run_r;
            const int nb = (bn + 31) >> 5;
            const int b = bi % WS_NBUF;
            if (first) {
                ws_pair_barrier(npt);                // the previous run's tile adds are complete
                if ((int64_t)r + 1 > flushed_upto) {
                    // rows pj <= r+1 can no longer be touched by this CTA
                    const int64_t lastrow = min((int64_t)r + 1, flushed_upto + rows - 2);
                    t_crumbs += bs_flush_rows(tile32, rows, cells, flushed_upto + 1, lastrow, W, cnt, npt, true);
                    flushed_upto = (int64_t)r + 1;
                    ws_pair_barrier(npt);            // retired ring slots may be reused by this run's tile add
                }
                rbase = (int)(((int64_t)r + 1) % rows);
                run_kmax = 0;
#pragma unroll
                for (int q = 0; q < NP; ++q)
#pragma unroll
                    for (int x = 0; x < 16; ++x) acc[q][x] = 0;
            }
            hx_mbar_wait(hx_smem_u32(&s_full[b]), (bi / WS_NBUF) & 1);
            const int *gk = gk0 + b * 32;
            const int bkm = __reduce_max_sync(0xffffffffu, lane < nb ? gk[lane] : 0);
            run_kmax = max(run_kmax, bkm);
#pragma unroll
            for (int q = 0; q < NP; ++q) {
                if (t2[q] < bkm) bs_accumulate(acc[q], planes_saddr + (uint32_t)(b * gb * kmax) * 16u, gk_saddr + b * 128u,
                                               t1[q], t2[q], nb, kmax);
            }
            __syncwarp();
            if (lane == 0) ws_mbar_arrive(hx_smem_u32(&s_empty[b]));
            if (last) {
#pragma unroll
                for (int q = 0; q < NP; ++q) {
                    if (t2[q] < run_kmax) {
                        int row = rbase + t2[q];
                        if (row >= rows) row -= rows;
                        const int d = t2[q] - t1[q];
                        uint4 *cell = tile + ((size_t)row * cells + (d - 1)) * 4;
#pragma unroll
                        for (int x = 0; x < 4; ++x) {
                            uint4 v = cell[x];
                            v.x += acc[q][4 * x + 0]; v.y += acc[q][4 * x + 1];
                            v.z += acc[q][4 * x + 2]; v.w += acc[q][4 * x + 3];
                            cell[x] = v;
                        }
                    }
                }
            }
        }
        ws_pair_barrier(npt);
        t_crumbs += bs_flush_rows(tile32, rows, cells, flushed_upto + 1, flushed_upto + rows - 1, W, cnt, npt, false);
    }
    if (errbits) atomicOr(err, (int)errbits);
    flush_totals(n_slices, t_crumbs + n_rcrumbs, (unsigned long long)n_codes - n_notcov, n_sent, totals);
}

}  // namespace

static std::atomic<bool> g_unsorted_seen{false};
bool hx_unsorted_seen() { return g_unsorted_seen.load(std::memory_order_relaxed); }
void hx_note_unsorted() { g_unsorted_seen.store(true, std::memory_order_relaxed); }

__global__ void k_flag_not(const int *__restrict__ in, int *__restrict__ out) {
    if (threadIdx.x == 0) *out = !*in;
}

static int launch_ingest(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off, const uint8_t *d_codes,
                         int64_t n_reads, int64_t *run_end, const int *ok);

int hx_launch_ingest(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off,
                     const uint8_t *d_codes, int64_t n_reads) {
    return launch_ingest(h, d_rank, d_off, d_codes, n_reads, nullptr, nullptr);
}

// The caller guarantees non-decreasing ranks and has filled run_end[N+1] (end of each rank's run of reads; the
// dense wire format's decode does both): no sortedness pre-pass, no generic fallback launch.  *ok (device) is
// non-zero when the chunk decoded consistently; the kernels do nothing otherwise.
int hx_launch_ingest_presorted(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off,
                               const uint8_t *d_codes, int64_t n_reads, int64_t *run_end, const int *ok) {
    return launch_ingest(h, d_rank, d_off, d_codes, n_reads, run_end, ok);
}

static int launch_ingest(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off, const uint8_t *d_codes,
                         int64_t n_reads, int64_t *run_end, const int *ok) {
    if (n_reads <= 0) return HX_OK;
    const bool presorted = run_end != nullptr;
    if (!presorted) run_end = h->d_run_end.p;
    const int sms = ingest_sm_budget(h);
    int *const verdict = &h->d_flags.p->ingest_sorted;      // the sortedness pre-pass writes its verdict here
    const int *sorted_flag = presorted ? ok : verdict;
    constexpr int GBLOCK = 256;
    const int64_t gwant = (n_reads + (GBLOCK / 32) - 1) / (GBLOCK / 32);
    const int ggrid = (int)(gwant < (int64_t)sms * 8 ? gwant : (int64_t)sms * 8);

    // crumbs in a read are all distinct cells, so W+1 bounds the SNPs per read
    const int kmax = h->W + 1;
    const bool bs_possible = kmax >= 2 && kmax <= BS_KMAX;
    const bool use_bs = (h->use.ingest_kernel == 2 || h->use.ingest_kernel == 4 || h->use.ingest_kernel == 5 || h->use.ingest_kernel == 6)
                            ? bs_possible : (h->use.ingest_kernel == 0 && bs_possible);
    // tensor-core kernel (ingest_umma.cu): default for rank-sorted reads of at most 32 SNPs
    // (auto: when a rank's run of reads is deep enough to fill MMAs - measured: 1000 reads per rank 0.42 vs 0.63 ms,
    // 20 reads per rank 0.25 vs 0.19 ms against the bit-sliced kernel)
    const bool use_umma = use_bs && hx_umma_possible(h) &&
                          (h->use.ingest_kernel == 6 || (h->use.ingest_kernel == 0 && n_reads >= 64 * ((int64_t)h->N + 1)));
    const bool use_long = !use_bs && (h->use.ingest_kernel == 3 || (h->use.ingest_kernel == 0 && kmax >= 2));
    // long-read tensor-core kernel (ingest_lumma.cu): default for wide reads unless its one-hot scratch would be huge
    const bool use_lumma = kmax >= 2 && (h->use.ingest_kernel == 7 ||
                                         (h->use.ingest_kernel == 0 && !use_bs &&
                                          hx_lumma_scratch_bytes(h, n_reads) <= ((int64_t)24 << 30)));

    // unsorted short reads: once this process has met some, the counting-sort tensor-core kernel is queued as the
    // fallback (it runs only if the pre-pass says "not sorted"); before that, and when its scratch would be huge, one
    // RED per pair (k1_pairs_red)
    const bool lumma_fallback = !presorted && use_bs && !use_lumma && h->use.ingest_kernel == 0 && hx_unsorted_seen() &&
                                hx_lumma_scratch_bytes(h, n_reads) <= ((int64_t)24 << 30);
    h->use.prepass_ran = !presorted && !use_lumma && (use_long || use_bs);
    HX_CUDA(cudaEventRecord(h->ev0, h->stream));
    if (use_lumma) {
        int rc = hx_launch_ingest_lumma(h, d_rank, d_off, d_codes, n_reads, presorted ? ok : nullptr);
        if (rc) return rc;
    } else if (use_long) {
        if (!presorted) {
            HX_CUDA(hx_fill_async(verdict, 1, sizeof(int), h->stream));     // non-zero = sorted
            k_prepass<<<(unsigned)((n_reads + 255) / 256), 256, 0, h->stream>>>(d_rank, n_reads, h->N, verdict,
                                                                                run_end, h->d_err.p);
            h->use.launches++;
        }
        int rc = hx_launch_ingest_long(h, d_rank, d_off, d_codes, n_reads, sorted_flag);
        if (rc) return rc;
        if (!presorted) {
            k1_pairs_red<GBLOCK><<<ggrid, GBLOCK, 0, h->stream>>>(d_rank, d_off, d_codes, n_reads, h->N, h->W,
                                                                  hx_cnt_ref(h), h->d_totals.p, h->d_err.p, sorted_flag, 0);
            h->use.launches++;
        }
    } else if (!use_bs) {
        k1_pairs_red<GBLOCK><<<ggrid, GBLOCK, 0, h->stream>>>(d_rank, d_off, d_codes, n_reads, h->N, h->W, hx_cnt_ref(h),
                                                              h->d_totals.p, h->d_err.p, sorted_flag, presorted ? 2 : 1);
        h->use.launches++;
    } else {
        if (!presorted) {
            // flag: non-zero = sorted; run_end: -1 = no reads of that rank (the tensor-core kernel walks it)
            k_prepass_init<<<(unsigned)((h->N + 2 + 255) / 256), 256, 0, h->stream>>>(verdict, run_end, use_umma ? h->N + 2 : 0);
            k_prepass<<<(unsigned)((n_reads + 255) / 256), 256, 0, h->stream>>>(d_rank, n_reads, h->N, verdict,
                                                                                run_end, h->d_err.p);
            h->use.launches += 2;
        }
        const int npairs = kmax * (kmax - 1) / 2;
        if (use_umma) {
            int rc = hx_launch_ingest_umma(h, d_rank, d_off, d_codes, n_reads, run_end, sorted_flag);
            if (rc) return rc;
        } else
        // measured (B200): the warp-specialised variant wins for wide reads (config 2: 0.097 vs 0.118 ms),
        // the barrier-phased one for narrow reads (config 3: 0.725 vs 0.751 ms)
        if (h->use.ingest_kernel == 5 || (h->use.ingest_kernel != 4 && kmax > 32)) {
            // warp-specialised: pw pair-owning warps + bw builder warps
            const int np = npairs > 512 ? 2 : 1;
            const int pw = ((npairs + np - 1) / np + 31) / 32;
            int bw = np == 1 && kmax <= 32 ? 20 - pw : 8;       // kmax <= 32: 20 warps, two CTAs per SM
            if (pw + bw > 32) bw = 32 - pw;
            const int block = (pw + bw) * 32;
            int gb = BS_GB;
            while (gb > 4 && WsLayout{kmax, gb}.bytes() > (size_t)((np == 1 ? 100 : 200) * 1024)) gb >>= 1;
            const size_t smem = WsLayout{kmax, gb}.bytes();
            const auto kern = ingest_kernel_for(h, [&](auto fused_t) {
                constexpr bool F = decltype(fused_t)::value;
                return np == 2 ? k1_bitsliced_ws<14, 2, 1024, 1, F>
                               : kmax > 32 ? k1_bitsliced_ws<14, 1, 1024, 1, F> : k1_bitsliced_ws<8, 1, 640, 2, F>;
            });
            unsigned grid;
            if (int rc = ingest_grid(kern, sms, block, smem, true, n_reads, &grid)) return rc;
            kern<<<grid, block, smem, h->stream>>>(d_rank, d_off, d_codes, n_reads, h->N, h->W, kmax, gb, pw, hx_cnt_ref(h),
                                                   h->d_totals.p, h->d_err.p, sorted_flag, run_end);
        } else {
        int gb = BS_GB;
        while (gb > 4 && BsLayout{kmax, gb}.bytes() > (size_t)200 * 1024) gb >>= 1;
        const size_t smem = BsLayout{kmax, gb}.bytes();
        const int np = npairs > 1024 ? 2 : 1;
        int block = ((npairs + np - 1) / np + 31) / 32 * 32;
        if (block < 128) block = 128;
        if (block > 1024) block = 1024;
        const auto kern = ingest_kernel_for(h, [&](auto fused_t) {
            constexpr bool F = decltype(fused_t)::value;
            return np == 2 ? k1_bitsliced<14, 2, 1024, 1, F>
                           : kmax > 32 ? k1_bitsliced<14, 1, 1024, 1, F> : k1_bitsliced<8, 1, 512, 2, F>;
        });
        unsigned grid;
        if (int rc = ingest_grid(kern, sms, block, smem, true, n_reads, &grid)) return rc;
        kern<<<grid, block, smem, h->stream>>>(d_rank, d_off, d_codes, n_reads, h->N, h->W, kmax, gb, hx_cnt_ref(h),
                                               h->d_totals.p, h->d_err.p, sorted_flag, run_end);
        }
        h->use.launches++;
        // fallback for unsorted input: runs only when the flag says the bit-sliced kernel declined
        if (lumma_fallback) {
            k_flag_not<<<1, 32, 0, h->stream>>>(verdict, &h->d_flags.p->fallback_go);
            h->use.launches++;
            int rc = hx_launch_ingest_lumma(h, d_rank, d_off, d_codes, n_reads, &h->d_flags.p->fallback_go);
            if (rc) return rc;
        } else if (!presorted) {
            k1_pairs_red<GBLOCK><<<ggrid, GBLOCK, 0, h->stream>>>(d_rank, d_off, d_codes, n_reads, h->N, h->W,
                                                                  hx_cnt_ref(h), h->d_totals.p, h->d_err.p, sorted_flag, 0);
            h->use.launches++;
        }
    }
    h->use.cnt_fresh = false;
    HX_CUDA(cudaGetLastError());
    HX_CUDA(cudaEventRecord(h->ev1, h->stream));
    h->use.ev_rec = true;
    return HX_OK;
}
