// K1 for long reads on the 5th-generation tensor cores (ONT-like, BASELINE configs[3]; any read wider than the
// bit-sliced / short-read tensor-core kernels take).  Same pair-expansion semantics as gretel/util.py:226-286.
//
// A read is a one-hot row x over the columns (site p, symbol a in A C G T N - _ and a spare): x[8p + a] = 1.  The
// counts it adds to every site pair (pi < pj) and symbol pair (a, b) are the entries of x^T x, so the whole band is
// C = X^T X restricted to 1 <= pj - pi <= W: an int8 GEMM with int32 accumulation (tcgen05.mma kind::i8, exact).
// Sites are cut into blocks of 16 (128 columns = the M / N of one MMA); the K of an MMA is a CHUNK of 32 reads.
//
//   k_l2_keys      per read: validate, key = (first block sb, blocks spanned), histogram of the keys
//   k_l2_pad       per first block: pad its reads up to a multiple of 32 -> chunks never mix first blocks
//   k_scan_*       exclusive scan of the padded histogram = where each key's reads go
//   k_l2_scatter   counting sort: perm[] = read indices ordered by (sb, span) (order inside a key is free: the
//                  counts are integer sums), so the 32 reads of a chunk start in the same block and end close together
//   k_l2_onehot    warp per chunk: the chunk's last block, sentinels, totals
//   k_l2_slabs     warp per (chunk, site block it touches), lane = read: writes the one-hot operand slab, 4 KB, laid out
//                  exactly as the MN-major UMMA operand (core matrix = 16 columns x 8 reads), so a slab is one 4 KB
//                  bulk copy away from the tensor core
//   k_l2_tiles     persistent CTAs over tiles (I = one block of 16 first sites, q = a pair of blocks of second sites):
//                  four producer warps (one per stage of the TMA/mbarrier ring) find the chunks that touch both (per
//                  first block the chunks are sorted by their last block: the sort's own offsets say where the
//                  reaching chunks start) and stream their slabs, up to 4 chunks per stage;
//                  one thread issues two M=128, N=128, K=32 MMAs per chunk into a double-buffered TMEM accumulator;
//                  8 epilogue warps read the finished accumulator (tcgen05.ld), turn it through shared memory
//                  into the band's cell order and add it to the band with coalesced read-modify-writes (plain stores
//                  into a freshly cleared matrix).  Every band cell has exactly one writer: no atomics.
//   k_l2_tiles2    the same over CTA pairs (cta_group::2, M = 256 across two SMs); opt-in, HX_LUMMA_PAIRS=1
// Rank-sortedness is not needed (the counting sort orders the reads itself).
#include <limits.h>
#include <stdlib.h>
#include <string.h>

#include "hx_internal.cuh"
#include "ingest_common.cuh"
#include "scan.cuh"

namespace {

constexpr int L2_G = 4;                             // chunks (of one first block) per pipeline stage
constexpr int L2_STAGES = 4;
constexpr int L2_EP_WARPS = 8;
constexpr int L2_PW = L2_STAGES;                        // producer warps: one per ring stage
constexpr int L2_THREADS = (L2_PW + 1 + L2_EP_WARPS) * 32;
constexpr int L2P_STAGES = 5;
constexpr int L2P_PW = L2P_STAGES;                      // the CTA-pair variant: its producer warps
constexpr int L2P_THREADS = (L2P_PW + 1 + L2_EP_WARPS) * 32;
constexpr uint32_t L2_SLAB = 4096;                 // one chunk x one block: 32 reads x 128 one-hot bytes
constexpr uint32_t L2_STAGE_BYTES = 3 * L2_G * L2_SLAB;   // A (first sites), B0, B1 (second sites), L2_G chunks each
constexpr int L2_STG_WORDS = 4 * 196;              // epilogue staging per warp: 4 second sites x 4 cells x 49 counters

#ifdef L2_PROFILE
__device__ unsigned long long l2_prof[16];
#endif

struct L2Geom {
    int N, W, NB, SP, nq;
    __host__ __device__ static L2Geom make(int N, int W) {
        L2Geom g;
        g.N = N; g.W = W;
        g.NB = (N >> 4) + 1;                        // sites 1..N live in blocks 0..N>>4
        g.SP = W / 16 + 2;                          // a read of k <= W+1 SNPs spans at most W/16 + 2 blocks
        g.nq = (g.SP + 1) / 2 + 1;                  // pairs of second-site blocks per first-site block
        return g;
    }
    __host__ __device__ int SPB() const { return SP + 1; }      // bins per first block: padding, then spans 0..SP-1
    __host__ __device__ int64_t n_bins() const { return (int64_t)NB * (SP + 1); }
};

// ---- sort keys ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_l2_keys(const int32_t *__restrict__ rank, const int64_t *__restrict__ off, int64_t n_reads, L2Geom g,
          int32_t *__restrict__ keys, int32_t *__restrict__ hist, int *__restrict__ err, const int *__restrict__ go) {
    if (go && !*go) return;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_reads) return;
    const int64_t k = off[i + 1] - off[i];
    const int r = rank[i];
    int key = -1;
    if (k >= 2) {                                                                    // util.py:230
        if (!read_fits(r, k, g.N, g.W)) atomicOr(err, 1);
        else {
            const int sb = (r + 1) >> 4, eb = (r + (int)k) >> 4;
            key = sb * g.SPB() + 1 + (eb - sb);
            atomicAdd(&hist[key], 1);
        }
    }
    keys[i] = key;
}

// bin 0 of every first block = the padding (in front of its shortest reads) that makes the block's read count a
// multiple of 32: bstart[sb*SPB + 1 + s] >> 5 is then exactly the first chunk holding a read that spans > s blocks
__global__ void k_l2_pad(int32_t *__restrict__ hist, L2Geom g, const int *__restrict__ go) {
    if (go && !*go) return;
    const int sb = blockIdx.x * blockDim.x + threadIdx.x;
    if (sb >= g.NB) return;
    int32_t *h = hist + (int64_t)sb * g.SPB();
    int s = 0;
    for (int j = 1; j <= g.SP; ++j) s += h[j];
    h[0] = (32 - (s & 31)) & 31;
}

__global__ void __launch_bounds__(256)
k_l2_scatter(const int32_t *__restrict__ keys, int64_t n_reads, const int32_t *__restrict__ bstart,
             int32_t *__restrict__ cursor, int32_t *__restrict__ perm, const int *__restrict__ go) {
    if (go && !*go) return;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_reads) return;
    const int key = keys[i];
    if (key < 0) return;
    perm[bstart[key] + atomicAdd(&cursor[key], 1)] = (int32_t)i;
}

// ---- one-hot operand slabs ----------------------------------------------------------------------------------
// Slab of (chunk c of first block sb, block sb+j) at onehot + (cs*SP + j*nch + (c-cs)) * 4096 with cs / nch = first
// chunk / number of chunks of sb; inside: [8 reads][16 columns] core matrices of 128 B,
// the 8 column groups of a block 128 B apart, the 4 groups of 8 reads 1024 B apart.
__global__ void __launch_bounds__(256)
k_l2_onehot(const int32_t *__restrict__ rank, const int64_t *__restrict__ off, const uint8_t *__restrict__ codes,
            const int32_t *__restrict__ perm, const int32_t *__restrict__ bstart, L2Geom g,
            uint8_t *__restrict__ onehot, int32_t *__restrict__ chunk_eb, const HxCnt cnt,
            unsigned long long *__restrict__ totals, int *__restrict__ err, const int *__restrict__ go) {
    if (go && !*go) return;
    const int lane = threadIdx.x & 31;
    const int64_t n_chunks = bstart[g.n_bins()] >> 5;
    const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    unsigned long long t_slices = 0, t_sent = 0;
    if (c < n_chunks) {
        const int idx = perm[c * 32 + lane];
        int r = 0, k = 0;
        int64_t o = 0;
        if (idx >= 0) {
            o = off[idx];
            k = (int)(off[idx + 1] - o);
            r = rank[idx];
        }
        const uint8_t *__restrict__ cd = codes + o;
        const int sb = __reduce_min_sync(0xffffffffu, idx >= 0 ? (r + 1) >> 4 : INT_MAX);
        const int eb = __reduce_max_sync(0xffffffffu, idx >= 0 ? (r + k) >> 4 : 0);
        if (lane == 0) chunk_eb[c] = eb;
        t_slices += idx >= 0;
        if (k >= 2) add_sentinels(cd, cd[0], r, k, g.N, g.W, cnt, t_sent);
    }
    flush_totals(t_slices, 0, 0, t_sent, totals);
}

// The slabs themselves: one warp per (chunk, site block) - a long-read chunk touches tens of blocks, and one warp per
// chunk left the GPU a third full of warps that each walked their reads serially (0.18 ms of a 1.1 ms ingestion).
// blockIdx.x = chunk, the 8 warps of a CTA take 8 consecutive blocks; lane = read.
__global__ void __launch_bounds__(256)
k_l2_slabs(const int32_t *__restrict__ rank, const int64_t *__restrict__ off, const uint8_t *__restrict__ codes,
           const int32_t *__restrict__ perm, const int32_t *__restrict__ bstart, L2Geom g,
           uint8_t *__restrict__ onehot, unsigned long long *__restrict__ totals, int *__restrict__ err,
           const int *__restrict__ go) {
    if (go && !*go) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n_chunks = bstart[g.n_bins()] >> 5;
    const int64_t c = blockIdx.x;
    if (c >= n_chunks) return;
    unsigned long long t_cov = 0;
    {
        const int idx = perm[c * 32 + lane];
        int r = 0, k = 0;
        int64_t o = 0;
        if (idx >= 0) {
            o = off[idx];
            k = (int)(off[idx + 1] - o);
            r = rank[idx];
        }
        const uint8_t *__restrict__ cd = codes + o;
        const int sb = __reduce_min_sync(0xffffffffu, idx >= 0 ? (r + 1) >> 4 : INT_MAX);
        const int eb = __reduce_max_sync(0xffffffffu, idx >= 0 ? (r + k) >> 4 : 0);
        const int b = sb + 8 * (int)blockIdx.y + warp;
        if (b <= eb) {
            // the slabs of a first block's chunks are stored block-major: a run of its chunks x one site block is contiguous
            const int64_t cs = bstart[(int64_t)sb * g.SPB()] >> 5, nch = (bstart[(int64_t)(sb + 1) * g.SPB()] >> 5) - cs;
            uint8_t *slab = onehot + ((size_t)cs * g.SP + (size_t)(c - cs) + (size_t)(b - sb) * (size_t)nch) * L2_SLAB +
                            (size_t)(lane >> 3) * 1024 + (size_t)(lane & 7) * 16;
            const int u0 = 16 * b - (r + 1);                       // position in my read of the block's first site
#pragma unroll
            for (int ch = 0; ch < 8; ++ch) {
                uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
                for (int s2 = 0; s2 < 2; ++s2) {
                    const int u = u0 + 2 * ch + s2;
                    if (u >= 0 && u < k) {
                        const unsigned a = cd[u];
                        if (a > 6) { atomicOr(err, 2); continue; }
                        t_cov += (a < 4 || a == HX_SYM_DEL);
                        if (a < 4) w[2 * s2] = 1u << (8 * a);
                        else w[2 * s2 + 1] = 1u << (8 * (a - 4));
                    }
                }
                *reinterpret_cast<uint4 *>(slab + ch * 128) = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
    }
    flush_totals(0, 0, t_cov, 0, totals);
}

// ---- tensor-core tiles -----------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t l2_desc(uint32_t saddr) {      // MN-major, no swizzle: LBO = 1024 (next 8 reads),
    uint64_t d = 0;                                                //                       SBO = 128 (next 16 columns)
    d |= (uint64_t)((saddr >> 4) & 0x3fffu);
    d |= (uint64_t)((1024u >> 4) & 0x3fffu) << 16;
    d |= (uint64_t)((128u >> 4) & 0x3fffu) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
// kind::i8, unsigned 8-bit A and B (both MN-major), int32 accumulators, M = 128, N = 128
constexpr uint32_t L2_IDESC = (2u << 4) | (1u << 15) | (1u << 16) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ void l2_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(L2_IDESC), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void l2_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void l2_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void l2_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void l2_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// One finished accumulator (128 TMEM lanes = 16 first sites x 8 symbols of block I; 256 columns = 32 second sites x 8
// symbols of blocks 2q, 2q+1) -> the band.  Called by every epilogue warp: quarter qd of the lanes (first sites 4qd..4qd+3),
// every (L2_EP_WARPS/4)-th group of four second sites starting at hsel.
template <bool FUSED, bool FRESH>
__device__ __forceinline__ void l2_epilogue_tile(uint32_t tmem_acc, int I, int q, int has, uint32_t *stg, int lane, int qd,
                                                 int hsel, const HxCnt &cnt, const L2Geom &g, unsigned long long &crumbs) {
    const int t1l = lane >> 3, a = lane & 7;
    const bool row_ok = a != HX_SYM_N && a != HX_SYM_GAP && a != 7;        // util.py:258: N and _ never come first
    const int my_stg = (3 - t1l) * 49 + a * 7;
    const int64_t W = g.W;
    const int pi = 16 * I + 4 * qd + t1l;
    for (int gq = hsel; gq < 8; gq += L2_EP_WARPS / 4) {
        const int half = gq >> 2;
        if (!((has >> half) & 1)) continue;
        uint32_t v[32];
        l2_ld32(tmem_acc + (uint32_t)gq * 32u + ((uint32_t)(qd * 32) << 16), v);
        const int pj0 = 16 * (2 * q + half) + (gq & 3) * 4;
        if (a != 7) {
#pragma unroll
            for (int t2l = 0; t2l < 4; ++t2l) {
                const bool ok = row_ok && pj0 + t2l > pi;
#pragma unroll
                for (int b = 0; b < 7; ++b) stg[t2l * 196 + my_stg + b] = ok ? v[t2l * 8 + b] : 0u;
            }
        }
        __syncwarp();
        // cells (pi, pj) of my quarter's four first sites are contiguous in band row pj: staging word i of
        // second site t2l lives at band word gbase + i
        uint32_t x[28];
#pragma unroll
        for (int t2l = 0; t2l < 4; ++t2l)
#pragma unroll
            for (int k = 0; k < 7; ++k) {
                const int i = k * 32 + lane;
                x[t2l * 7 + k] = i < 196 ? stg[t2l * 196 + i] : 0u;
            }
        __syncwarp();
        if (!FUSED && FRESH) {
            // the band is still all zero (first ingestion into this matrix): plain stores, no loads.  Where the
            // warp's four cells lie inside the band every word is written, zeros too (whole sectors: nothing
            // for L2 to fetch); the sentinel cells (pi = 0, pj = N+1) are never touched.
            const int pi_lo = 16 * I + 4 * qd;
#pragma unroll
            for (int t2l = 0; t2l < 4; ++t2l) {
                const int64_t pj = pj0 + t2l;
                const bool full = pi_lo >= 1 && pj <= g.N && pj - (pi_lo + 3) >= 1 && pj - pi_lo <= W;
                uint32_t *gb = cnt.local + (pj * W + pj - 16 * I - 4 * qd - 4) * HX_CELL + lane;
#pragma unroll
                for (int k = 0; k < 7; ++k) {
                    const uint32_t xv = x[t2l * 7 + k];
                    if (xv || (full && k * 32 + lane < 196)) gb[k * 32] = xv;
                    crumbs += xv;
                }
            }
        } else if (!FUSED) {
            uint32_t old[28];
#pragma unroll
            for (int t2l = 0; t2l < 4; ++t2l) {
                const int64_t pj = pj0 + t2l;
                uint32_t *gb = cnt.local + (pj * W + pj - 16 * I - 4 * qd - 4) * HX_CELL + lane;
#pragma unroll
                for (int k = 0; k < 7; ++k)
                    if (x[t2l * 7 + k]) old[t2l * 7 + k] = gb[k * 32];
            }
#pragma unroll
            for (int t2l = 0; t2l < 4; ++t2l) {
                const int64_t pj = pj0 + t2l;
                uint32_t *gb = cnt.local + (pj * W + pj - 16 * I - 4 * qd - 4) * HX_CELL + lane;
#pragma unroll
                for (int k = 0; k < 7; ++k)
                    if (x[t2l * 7 + k]) {
                        gb[k * 32] = old[t2l * 7 + k] + x[t2l * 7 + k];
                        crumbs += x[t2l * 7 + k];
                    }
            }
        } else {
#pragma unroll
            for (int t2l = 0; t2l < 4; ++t2l) {
                const int64_t pj = pj0 + t2l;
                uint32_t *base = cnt.peer[pj / cnt.rows_per];
                uint32_t *gb = base + (pj * W + pj - 16 * I - 4 * qd - 4) * HX_CELL + lane;
#pragma unroll
                for (int k = 0; k < 7; ++k)
                    if (x[t2l * 7 + k]) {
                        atomicAdd(gb + k * 32, x[t2l * 7 + k]);
                        crumbs += x[t2l * 7 + k];
                    }
            }
        }
    }
}

// stage meta = (I, q, flags): flags 1 = B0 present, 2 = B1 present, 4 = last chunk of the tile, 8 = exit

template <bool FUSED, bool FRESH>
__global__ void __launch_bounds__(L2_THREADS, 1)
k_l2_tiles(const uint8_t *__restrict__ onehot, const int32_t *__restrict__ bstart, L2Geom g, const HxCnt cnt_in,
           unsigned long long *__restrict__ totals, const int *__restrict__ go) {
    extern __shared__ __align__(1024) uint8_t l2_smem[];
    __shared__ __align__(8) unsigned long long s_full[L2_STAGES], s_empty[L2_STAGES], s_acc_full[2], s_acc_empty[2];
    __shared__ __align__(8) int s_meta[L2_STAGES][2];
    __shared__ int4 s_runs[L2_STAGES][64];            // per producer warp: the runs of chunks of the tile being sent
    __shared__ int2 s_pend[L2_STAGES][L2_G];
    __shared__ volatile int s_tile[2][4];             // (I, q, halves present, exit) of the tile in each accumulator
    __shared__ uint32_t s_tmem;
    if (go && !*go) return;
    const HxCnt cnt = cnt_in.for_build<FUSED>();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t stage0 = hx_smem_u32(l2_smem);
    uint32_t *const staging = reinterpret_cast<uint32_t *>(l2_smem + (size_t)L2_STAGES * L2_STAGE_BYTES);

    if (threadIdx.x == 0) {
        for (int s = 0; s < L2_STAGES; ++s) {
            hx_mbar_init(hx_smem_u32(&s_full[s]), 1);
            hx_mbar_init(hx_smem_u32(&s_empty[s]), 1);
        }
        for (int s = 0; s < 2; ++s) {
            hx_mbar_init(hx_smem_u32(&s_acc_full[s]), 1);
            hx_mbar_init(hx_smem_u32(&s_acc_empty[s]), L2_EP_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(hx_smem_u32(&s_tmem)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    l2_fence_before();
    __syncthreads();
    l2_fence_after();
    const uint32_t tmem_base = s_tmem;
    const int SP = g.SP;
    unsigned long long crumbs = 0;

    if (warp < L2_PW) {
        // ============================== producers ======================================
        // A lone warp needs several hundred cycles per stage (barrier wait, meta, three bulk copies), more than the
        // MMAs of the stage take, so there is one producer warp per ring stage: every warp walks the same static tile
        // list and derives the same sequence of pieces (runs of up to L2_G chunks of one first block); warp w sends the
        // pieces k = w (mod L2_PW), always into stage w.
        const int64_t n_tiles = (int64_t)g.NB * g.nq;
        const int SPB = g.SPB();
        const uint32_t bar_full = hx_smem_u32(&s_full[warp]), bar_empty = hx_smem_u32(&s_empty[warp]);
        const uint32_t dst0 = stage0 + (uint32_t)warp * L2_STAGE_BYTES;
        int4 *const runs = s_runs[warp];
        int2 *const pend = s_pend[warp];                 // the stage being collected: up to L2_G chunks (slab of block I, nch | b1)
        unsigned ph = 0, turn = 0;                       // phase of my stage; whose stage comes next
        int n_pend = 0, p_I = 0, p_q = 0;
        // a stage = up to L2_G chunks of the tile, whatever first block they belong to: one 4 KB bulk copy per chunk
        // and operand (lane = 3 * slot + operand)
        auto emit = [&](int last) {
            if (turn == (unsigned)warp) {
                const int b0 = 2 * p_q >= p_I;
                __syncwarp();
                const int slot = lane / 3, op = lane - 3 * slot;
                int2 c = make_int2(0, 0);
                if (slot < n_pend) c = pend[slot];
                const int b1 = (unsigned)c.y >> 31, nch = c.y & 0x7fffffff;
                const bool mine = slot < n_pend && (op == 0 || (op == 1 ? b0 : b1));
                const unsigned b1mask = __ballot_sync(0xffffffffu, slot < n_pend && op == 2 && b1);   // bit 3*slot+2
                const unsigned n_copies = __popc(__ballot_sync(0xffffffffu, mine));
                if (lane == 0) {
                    hx_mbar_wait(bar_empty, ph ^ 1);
                    // meta: I | q, chunks, B0 present, last, per-chunk "B1 present"
                    unsigned b1bits = 0;
#pragma unroll
                    for (int i = 0; i < L2_G; ++i) b1bits |= ((b1mask >> (3 * i + 2)) & 1u) << i;
                    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(hx_smem_u32(&s_meta[warp][0])), "r"(p_I),
                                 "r"(p_q | (n_pend << 20) | ((b0 | (last << 2)) << 24) | (b1bits << 28))
                                 : "memory");
#ifdef L2_NOCOPY
                    hx_mbar_expect_tx(bar_full, 0);
#else
                    hx_mbar_expect_tx(bar_full, L2_SLAB * n_copies);
#endif
                }
                __syncwarp();
#ifdef L2_NOCOPY
                if (false) {
#else
                if (mine) {
#endif
                    const int slab = c.x + (op ? (2 * p_q - p_I + op - 1) * nch : 0);
                    hx_bulk_g2s(dst0 + (uint32_t)(op * L2_G + slot) * L2_SLAB, onehot + (size_t)slab * L2_SLAB, L2_SLAB, bar_full);
                }
                ph ^= 1;
            }
            if (++turn == L2_PW) turn = 0;
            n_pend = 0;
        };
        const unsigned lt = (1u << lane) - 1u;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            const int I = (int)(t / g.nq), q = (I >> 1) + (int)(t % g.nq);
            const int jmax = min(I + SP - 1, g.NB - 1);
            if (2 * q > jmax) continue;
            const int jlo = max(2 * q, I);
            // first blocks whose reads can reach jlo: sb >= jlo - (SP-1); they must start at or before I
            const int sb_lo = max(0, jlo - SP + 1);
            for (int sb0 = sb_lo; sb0 <= I; sb0 += 32) {
                const int sb = sb0 + lane;
                int first = 0, end = 0, cb1 = 0, cs = 0;
                if (sb <= I) {
                    // the reads of a first block are sorted by the blocks they span: those reaching block j are a suffix
                    const int32_t *__restrict__ bs = bstart + (int64_t)sb * SPB;
                    const int d1 = 2 * q + 1 - sb;
                    cs = bs[0] >> 5;
                    first = bs[1 + jlo - sb] >> 5;
                    end = bs[SPB] >> 5;
                    cb1 = d1 < SP ? max(bs[1 + d1] >> 5, first) : end;       // chunks from cb1 on reach block 2q+1
                }
                // every first block gives up to two runs of chunks: [first, cb1) without and [cb1, end) with block 2q+1
                // (the slabs of block 2q+1 only exist from chunk cb1 on); the runs go to shared memory in lane order
                const int nch = end - cs;
                const int slab0 = cs * SP + (I - sb) * nch - cs;           // + chunk index = slab of (chunk, block I)
                const unsigned mA = __ballot_sync(0xffffffffu, first < cb1), mB = __ballot_sync(0xffffffffu, cb1 < end);
                int at = __popc(mA & lt) + __popc(mB & lt);
                if (first < cb1) runs[at++] = make_int4(slab0 + first, nch, cb1 - first, 0);
                if (cb1 < end) runs[at] = make_int4(slab0 + cb1, nch, end - cb1, 1);
                const int n_runs = __popc(mA) + __popc(mB);
                __syncwarp();
                for (int j = 0; j < n_runs; ++j) {
                    const int4 run = runs[j];
                    for (int o = 0; o < run.z; ++o) {
                        if (n_pend == L2_G) emit(0);
                        if (turn == (unsigned)warp && lane == 0) pend[n_pend] = make_int2(run.x + o, run.y | (run.w << 31));
                        ++n_pend; p_I = I; p_q = q;
                    }
                }
                __syncwarp();
            }
            if (n_pend) emit(1);
        }
        if (turn == (unsigned)warp && lane == 0) {                   // the warp whose turn it is tells the MMA thread to stop
            hx_mbar_wait(bar_empty, ph ^ 1);
            asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(hx_smem_u32(&s_meta[warp][0])), "r"(0), "r"(8 << 24) : "memory");
            ws_mbar_arrive(bar_full);
        }
    } else if (warp == L2_PW) {
        // ============================== MMA issue ======================================
        if (lane == 0) {
            unsigned stage = 0, ph = 0, acc = 0, acc_ph[2] = {0, 0};
            bool new_tile = true;
            int has = 0;
#ifdef L2_PROFILE
            unsigned long long pw = 0, pi_ = 0, pa = 0, pn = 0, pm = 0;
            const long long t_begin = clock64();
#endif
            for (;;) {
#ifdef L2_PROFILE
                const long long c0 = clock64();
#endif
                hx_mbar_wait(hx_smem_u32(&s_full[stage]), ph);
#ifdef L2_PROFILE
                const long long c1 = clock64(); pw += c1 - c0; pn++;
#endif
                int m_I, m_w;
                asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(m_I), "=r"(m_w) : "r"(hx_smem_u32(&s_meta[stage][0])) : "memory");
                const int m_q = m_w & 0xfffff, m_flags = (m_w >> 24) & 15, n = (m_w >> 20) & 15;
                const unsigned m_b1 = (unsigned)m_w >> 28;
                if (m_flags & 8) {
#ifdef L2_PROFILE
                    atomicAdd(&l2_prof[0], pw); atomicAdd(&l2_prof[1], pi_); atomicAdd(&l2_prof[2], pa); atomicAdd(&l2_prof[3], pn); atomicAdd(&l2_prof[4], pm);
                    atomicAdd(&l2_prof[5], (unsigned long long)(clock64() - t_begin));
#endif
                    hx_mbar_wait(hx_smem_u32(&s_acc_empty[acc]), acc_ph[acc] ^ 1);
                    s_tile[acc][3] = 1;
                    ws_mbar_arrive(hx_smem_u32(&s_acc_full[acc]));
                    break;
                }
                if (new_tile) {
#ifdef L2_PROFILE
                    const long long c2 = clock64();
#endif
                    hx_mbar_wait(hx_smem_u32(&s_acc_empty[acc]), acc_ph[acc] ^ 1);
#ifdef L2_PROFILE
                    pa += clock64() - c2;
#endif
                    new_tile = false;
                    has = 0;
                }
#ifdef L2_PROFILE
                const long long c3 = clock64();
#endif
                l2_fence_after();
                const uint32_t sa = stage0 + stage * L2_STAGE_BYTES;
                const uint32_t d = tmem_base + acc * 256u;
                const uint64_t da = l2_desc(sa), db0 = l2_desc(sa + L2_G * L2_SLAB), db1 = l2_desc(sa + 2 * L2_G * L2_SLAB);
                for (int i = 0; i < n; ++i) {                       // the next chunk's slab is 4096 B = 256 descriptor units on
                    const uint64_t o = (uint64_t)(i * (int)(L2_SLAB >> 4));
                    if (m_flags & 1) { l2_mma(d, da + o, db0 + o, has & 1); has |= 1; }
                    if ((m_b1 >> i) & 1) { l2_mma(d + 128u, da + o, db1 + o, (has >> 1) & 1); has |= 2; }
                }
#ifdef L2_PROFILE
                pi_ += clock64() - c3; pm += n * ((m_flags & 1) != 0) + __popc(m_b1);
#endif
                l2_commit(hx_smem_u32(&s_empty[stage]));
                if (m_flags & 4) {
                    s_tile[acc][0] = m_I; s_tile[acc][1] = m_q; s_tile[acc][2] = has; s_tile[acc][3] = 0;
                    asm volatile("fence.acq_rel.cta;" ::: "memory");
                    l2_commit(hx_smem_u32(&s_acc_full[acc]));
                    acc_ph[acc] ^= 1;
                    acc ^= 1;
                    new_tile = true;
                }
                if (++stage == L2_STAGES) { stage = 0; ph ^= 1; }
            }
        }
    } else {
        // ============================== epilogue ======================================
        const int ew = warp - (L2_PW + 1), qd = warp & 3, hsel = ew >> 2;
        uint32_t *const stg = staging + (size_t)ew * L2_STG_WORDS;
        unsigned acc = 0, acc_ph[2] = {0, 0};
        for (;;) {
            ws_mbar_wait_sleep(hx_smem_u32(&s_acc_full[acc]), acc_ph[acc]);
            acc_ph[acc] ^= 1;
            l2_fence_after();
            if (s_tile[acc][3]) break;
            const int I = s_tile[acc][0], q = s_tile[acc][1], has = s_tile[acc][2];
            l2_epilogue_tile<FUSED, FRESH>(tmem_base + acc * 256u, I, q, has, stg, lane, qd, hsel, cnt, g, crumbs);
            l2_fence_before();
            __syncwarp();
            if (lane == 0) ws_mbar_arrive(hx_smem_u32(&s_acc_empty[acc]));
            acc ^= 1;
        }
    }
    l2_fence_before();
    flush_totals(0, crumbs, 0, 0, totals);                            // barriers inside
    if (warp == 0) {
        l2_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ---- the same tiles on CTA pairs (cta_group::2) ---------------------------------------------------------------
// An M=N=128, K=32 int8 MMA reads 8 KB of operands from shared memory in its 64 cycles - all of the 128 B/clk there
// is - so in k_l2_tiles every byte TMA refills comes out of the MMA rate (measured: ~140 cycles per MMA).  Two CTAs of a
// cluster (the two SMs of a TPC) run ONE M=256, N=256 MMA per chunk instead: CTA r holds the A rows of first-site block
// 2Ip+r and the B columns of second-site block 2q+r, the hardware shares the halves, and each SM's shared memory sees
// 4 KB of fills + 4 KB of operand reads per 128x128x32 of work instead of 6 + 8.
//   * both CTAs walk the same static tile list (tile = pair of first blocks x pair of second blocks) and derive the
//     same runs of chunks from the sort offsets; each loads its own two slabs per chunk (a zero slab where the chunk
//     has none for that block) and signals its own `full` barrier;
//   * warp 1 of the second CTA forwards `full` to the leader (remote mbarrier arrive); the leader's MMA thread waits for
//     both, issues, and tcgen05.commit-multicasts `empty` (stage reusable) and `acc_full` (tile done) to both CTAs;
//   * each CTA's epilogue warps drain their own 128 TMEM lanes exactly as in k_l2_tiles and release the accumulator
//     on a local barrier and on the leader's pair barrier.
constexpr int L2P_G = 4;
constexpr uint32_t L2P_STAGE_BYTES = 2 * L2P_G * L2_SLAB;        // A slabs, B slabs
constexpr uint32_t L2P_IDESC = (2u << 4) | (1u << 15) | (1u << 16) | ((256u >> 3) << 17) | ((256u >> 4) << 24);

__device__ __forceinline__ uint32_t l2_mapa(uint32_t addr, uint32_t cta) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta));
    return r;
}
__device__ __forceinline__ void l2_remote_arrive(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void l2_wait_cluster(uint32_t bar, uint32_t parity) {
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) break;
    }
}
__device__ __forceinline__ void l2_mma2(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(L2P_IDESC), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void l2_commit2(uint32_t bar) {       // arrives on the barrier at this offset in BOTH CTAs
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"((uint16_t)3)
                 : "memory");
}
__device__ __forceinline__ void l2_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <bool FRESH>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(L2P_THREADS, 1)
k_l2_tiles2(const uint8_t *__restrict__ onehot, const uint8_t *__restrict__ zero_slabs, const int32_t *__restrict__ bstart,
            L2Geom g, const HxCnt cnt_in, unsigned long long *__restrict__ totals, const int *__restrict__ go) {
    extern __shared__ __align__(1024) uint8_t l2_smem[];
    __shared__ __align__(8) unsigned long long s_full[L2P_STAGES], s_empty[L2P_STAGES], s_peer_full[L2P_STAGES];
    __shared__ __align__(8) unsigned long long s_acc_full[2], s_acc_empty_local[2], s_acc_empty_pair[2], s_tile_ready[2];
    __shared__ __align__(8) int s_meta[L2P_STAGES][2];
    __shared__ int4 s_runs[L2P_STAGES][128];
    __shared__ int4 s_pend[L2P_STAGES][L2P_G];
    __shared__ volatile int s_tile[2][4];
    __shared__ uint32_t s_tmem;
    if (go && !*go) return;                              // (uniform over the cluster)
    const HxCnt cnt = cnt_in.for_build<false>();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
    const uint32_t stage0 = hx_smem_u32(l2_smem);
    uint32_t *const staging = reinterpret_cast<uint32_t *>(l2_smem + (size_t)L2P_STAGES * L2P_STAGE_BYTES);

    if (threadIdx.x == 0) {
        for (int s = 0; s < L2P_STAGES; ++s) {
            hx_mbar_init(hx_smem_u32(&s_full[s]), 1);
            hx_mbar_init(hx_smem_u32(&s_empty[s]), 1);
            hx_mbar_init(hx_smem_u32(&s_peer_full[s]), 1);
        }
        for (int s = 0; s < 2; ++s) {
            hx_mbar_init(hx_smem_u32(&s_acc_full[s]), 1);
            hx_mbar_init(hx_smem_u32(&s_acc_empty_local[s]), L2_EP_WARPS);
            hx_mbar_init(hx_smem_u32(&s_acc_empty_pair[s]), 2 * L2_EP_WARPS);
            hx_mbar_init(hx_smem_u32(&s_tile_ready[s]), 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(hx_smem_u32(&s_tmem)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    l2_fence_before();
    __syncthreads();
    l2_cluster_sync();                                    // the partner's barriers exist before anything arrives on them
    l2_fence_after();
    const uint32_t tmem_base = s_tmem;
    const int SP = g.SP;
    unsigned long long crumbs = 0;

    if (warp < L2P_PW) {
        // ============================== producers (both CTAs, identical tile and chunk lists) ===================
        // one warp per ring stage, as in k_l2_tiles; a stage = up to L2P_G chunks, two 4 KB bulk copies per chunk here
        // (lane = 2 * slot + operand: my A block, my B block; a zero slab where the chunk has none for that block)
        const int nq = g.nq;
        const int64_t n_tiles = (int64_t)((g.NB + 1) >> 1) * nq;
        const int SPB = g.SPB();
        const uint32_t bar_full = hx_smem_u32(&s_full[warp]), bar_empty = hx_smem_u32(&s_empty[warp]);
        const uint32_t dst0 = stage0 + (uint32_t)warp * L2P_STAGE_BYTES;
        int4 *const runs = s_runs[warp];
        int4 *const pend = s_pend[warp];                 // chunk: slab of its first block, nch, first block, reaches 2q+1
        const uint32_t peer_full_at_leader = l2_mapa(hx_smem_u32(&s_peer_full[warp]), 0);
        unsigned ph = 0, gturn = 0;                      // phase of my stage; (stages sent so far by all warps) mod L2P_PW
        int n_pend = 0, p_Ip = 0, p_q = 0;
        auto emit = [&](int last) {                      // called by the stage's owner only
            {
                __syncwarp();
                const int slot = lane >> 1, op = lane & 1;
                const bool mine = slot < n_pend;
                if (lane == 0) {
                    l2_wait_cluster(bar_empty, ph ^ 1);
                    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(hx_smem_u32(&s_meta[warp][0])), "r"(p_Ip),
                                 "r"(p_q | (n_pend << 20) | (last << 24))
                                 : "memory");
                    hx_mbar_expect_tx(bar_full, 2 * L2_SLAB * (uint32_t)n_pend);
                }
                __syncwarp();
                if (mine) {
                    const int4 c = pend[slot];                       // x, nch, sb, b1
                    const int blk = op == 0 ? 2 * p_Ip + (int)rank : 2 * p_q + (int)rank;
                    // does this chunk have a slab for blk?  (its first block is at or before it and it reaches it)
                    bool have = c.z <= blk;
                    if (rank == 1) have = have && (op == 0 ? (p_q > p_Ip || c.w) : (c.w != 0));
                    const uint8_t *src = have ? onehot + ((size_t)c.x + (size_t)(blk - c.z) * c.y) * L2_SLAB : zero_slabs;
                    hx_bulk_g2s(dst0 + (uint32_t)(op * L2P_G + slot) * L2_SLAB, src, L2_SLAB, bar_full);
                }
                // the second CTA tells the leader when its half of the stage has landed: each producer warp forwards its
                // own stage (a remote arrive costs its issuer several hundred cycles - one forwarding thread for all
                // stages paced the whole pipeline)
                if (rank == 1 && lane == 0) {
                    l2_wait_cluster(bar_full, ph);
                    l2_remote_arrive(peer_full_at_leader);
                }
                ph ^= 1;
            }
        };
        const unsigned lt = (1u << lane) - 1u;
        for (int64_t t = pair; t < n_tiles; t += n_pairs) {
            const int Ip = (int)(t / nq), q = Ip + (int)(t % nq);
            const int I0 = 2 * Ip, I1 = min(I0 + 1, g.NB - 1);
            const int jmax = min(I1 + SP - 1, g.NB - 1);
            if (2 * q > jmax) continue;
            const int jlo = 2 * q;                                  // q >= Ip: the second blocks start at or after I0
            const int sb_lo = max(0, jlo - SP + 1);
            // the tile's runs of chunks (two per first block, SP <= 64 first blocks: at most 128), in shared memory
            int n_runs = 0;
            for (int sb0 = sb_lo; sb0 <= I1; sb0 += 32) {
                const int sb = sb0 + lane;
                int first = 0, end = 0, cb1 = 0, cs = 0;
                if (sb <= I1) {
                    const int32_t *__restrict__ bs = bstart + (int64_t)sb * SPB;
                    const int d1 = 2 * q + 1 - sb;
                    cs = bs[0] >> 5;
                    first = bs[1 + max(jlo - sb, 0)] >> 5;
                    end = bs[SPB] >> 5;
                    cb1 = d1 <= 0 ? first : (d1 < SP ? max(bs[1 + d1] >> 5, first) : end);
                }
                const int nch = end - cs;
                const int x0 = cs * SP - cs;                        // + chunk index = slab of (chunk, block sb)
                const unsigned mA = __ballot_sync(0xffffffffu, first < cb1), mB = __ballot_sync(0xffffffffu, cb1 < end);
                int at = n_runs + __popc(mA & lt) + __popc(mB & lt);
                if (first < cb1) runs[at++] = make_int4(x0 + first, nch, cb1 - first, sb << 1);
                if (cb1 < end) runs[at] = make_int4(x0 + cb1, nch, end - cb1, (sb << 1) | 1);
                n_runs += __popc(mA) + __popc(mB);
            }
            __syncwarp();
            // chunk c of the tile = chunk (c - start[r]) of run r: lane j keeps runs 4j .. 4j+3 and their starts
            int4 my[4];
            int st[5];
            st[0] = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                my[i] = 4 * lane + i < n_runs ? runs[4 * lane + i] : make_int4(0, 0, 0, 0);
                st[i + 1] = st[i] + my[i].z;
            }
            int incl = st[4];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const int base = incl - st[4];
            const int T = __shfl_sync(0xffffffffu, incl, 31);
            const int n_st = (T + L2P_G - 1) / L2P_G;
            __syncwarp();
            // my stages of this tile: the global stage counter decides whose turn it is
            for (int k = (int)((unsigned)(warp + L2P_PW - (int)gturn) % L2P_PW); k < n_st; k += L2P_PW) {
                const int n_slots = min(L2P_G, T - k * L2P_G);
#pragma unroll
                for (int sl = 0; sl < L2P_G; ++sl) {
                    const int c = k * L2P_G + sl - base;             // position among my runs' chunks
                    if (sl < n_slots && c >= 0 && c < st[4]) {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            if (c >= st[i] && c < st[i + 1])
                                pend[sl] = make_int4(my[i].x + (c - st[i]), my[i].y, my[i].w >> 1, my[i].w & 1);
                    }
                }
                n_pend = n_slots; p_Ip = Ip; p_q = q;
                emit(k == n_st - 1);
            }
            gturn = (gturn + (unsigned)n_st) % L2P_PW;
        }
        if (gturn == (unsigned)warp && lane == 0) {                  // the warp whose turn it is tells warp L2P_PW to stop
            l2_wait_cluster(bar_empty, ph ^ 1);
            asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(hx_smem_u32(&s_meta[warp][0])), "r"(0), "r"(8 << 24) : "memory");
            ws_mbar_arrive(bar_full);
        }
    } else if (warp == L2P_PW) {
        // ============================== MMA issue (leader) / forwarding (second CTA) ===========================
        if (lane == 0) {
            unsigned stage = 0, ph = 0, acc = 0, acc_ph[2] = {0, 0};
            bool new_tile = true, first = true;
            const uint32_t acc_empty = hx_smem_u32(rank == 0 ? &s_acc_empty_pair[0] : &s_acc_empty_local[0]);
#ifdef L2_PROFILE
            unsigned long long pw = 0, pp = 0, pi_ = 0, pa = 0, pn = 0, pm = 0;
            const long long t_begin = clock64();
#endif
            for (;;) {
#ifdef L2_PROFILE
                const long long c0 = clock64();
#endif
                l2_wait_cluster(hx_smem_u32(&s_full[stage]), ph);
#ifdef L2_PROFILE
                pw += clock64() - c0; pn++;
#endif
                int m_Ip, m_w;
                asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(m_Ip), "=r"(m_w) : "r"(hx_smem_u32(&s_meta[stage][0])) : "memory");
                const int m_q = m_w & 0xfffff, m_flags = m_w >> 24, n = (m_w >> 20) & 15;
                if (m_flags & 8) {
#ifdef L2_PROFILE
                    if (rank == 0) { atomicAdd(&l2_prof[0], pw); atomicAdd(&l2_prof[1], pi_); atomicAdd(&l2_prof[2], pa); atomicAdd(&l2_prof[3], pn); atomicAdd(&l2_prof[4], pm);
                    atomicAdd(&l2_prof[5], (unsigned long long)(clock64() - t_begin)); atomicAdd(&l2_prof[6], pp); }
#endif
                    l2_wait_cluster(acc_empty + 8u * acc, acc_ph[acc] ^ 1);
                    s_tile[acc][3] = 1;
                    ws_mbar_arrive(hx_smem_u32(&s_tile_ready[acc]));
                    ws_mbar_arrive(hx_smem_u32(&s_acc_full[acc]));
                    break;
                }
                if (new_tile) {
#ifdef L2_PROFILE
                    const long long c2 = clock64();
#endif
                    l2_wait_cluster(acc_empty + 8u * acc, acc_ph[acc] ^ 1);
#ifdef L2_PROFILE
                    pa += clock64() - c2;
#endif
                    new_tile = false;
                    first = true;
                }
                if (m_flags & 1) {                                   // the tile's last stage: say which tile it was
                    s_tile[acc][0] = 2 * m_Ip + (int)rank; s_tile[acc][1] = m_q; s_tile[acc][2] = 3; s_tile[acc][3] = 0;
                    ws_mbar_arrive(hx_smem_u32(&s_tile_ready[acc]));
                }
                if (rank == 0) {
#ifdef L2_PROFILE
                    const long long c3 = clock64();
#endif
                    l2_wait_cluster(hx_smem_u32(&s_peer_full[stage]), ph);
#ifdef L2_PROFILE
                    const long long c4 = clock64(); pp += c4 - c3;
#endif
                    l2_fence_after();
                    const uint32_t sa = stage0 + stage * L2P_STAGE_BYTES;
                    const uint32_t d = tmem_base + acc * 256u;
                    const uint64_t da = l2_desc(sa), db = l2_desc(sa + L2P_G * L2_SLAB);
                    for (int i = 0; i < n; ++i) {
                        const uint64_t o = (uint64_t)(i * (int)(L2_SLAB >> 4));
                        l2_mma2(d, da + o, db + o, first ? 0u : 1u);
                        first = false;
                    }
#ifdef L2_PROFILE
                    pi_ += clock64() - c4; pm += n;
#endif
                    l2_commit2(hx_smem_u32(&s_empty[stage]));
                    if (m_flags & 1) l2_commit2(hx_smem_u32(&s_acc_full[acc]));
                }
                if (m_flags & 1) {
                    acc_ph[acc] ^= 1;
                    acc ^= 1;
                    new_tile = true;
                }
                if (++stage == L2P_STAGES) { stage = 0; ph ^= 1; }
            }
        }
    } else {
        // ============================== epilogue (each CTA drains its own 128 TMEM lanes) ======================
        const int ew = warp - (L2P_PW + 1), qd = warp & 3, hsel = ew >> 2;
        uint32_t *const stg = staging + (size_t)ew * L2_STG_WORDS;
        const uint32_t pair_bar0 = l2_mapa(hx_smem_u32(&s_acc_empty_pair[0]), 0);
        unsigned acc = 0, acc_ph[2] = {0, 0};
        for (;;) {
            l2_wait_cluster(hx_smem_u32(&s_acc_full[acc]), acc_ph[acc]);
            l2_wait_cluster(hx_smem_u32(&s_tile_ready[acc]), acc_ph[acc]);      // (warp L2P_PW has said which tile it is)
            acc_ph[acc] ^= 1;
            l2_fence_after();
            if (s_tile[acc][3]) break;
            const int I = s_tile[acc][0], q = s_tile[acc][1];
            if (I < g.NB)
                l2_epilogue_tile<false, FRESH>(tmem_base + acc * 256u, I, q, 3, stg, lane, qd, hsel, cnt, g, crumbs);
            l2_fence_before();
            __syncwarp();
            if (lane == 0) {
                ws_mbar_arrive(hx_smem_u32(&s_acc_empty_local[acc]));
                l2_remote_arrive(pair_bar0 + 8u * acc);
            }
            acc ^= 1;
        }
    }
    l2_fence_before();
    flush_totals(0, crumbs, 0, 0, totals);                            // barriers inside
    l2_cluster_sync();                                                // nothing of the partner is still on its way here
    if (warp == 0) {
        l2_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

}  // namespace

#ifdef L2_PROFILE
extern "C" int hx_debug_l2_prof(unsigned long long *out, int reset) {
    if (cudaMemcpyFromSymbol(out, l2_prof, sizeof(unsigned long long) * 16) != cudaSuccess) return -1;
    if (reset) {
        unsigned long long z[16] = {0};
        cudaMemcpyToSymbol(l2_prof, z, sizeof(z));
    }
    return 0;
}
#endif

// Scratch owned by the matrix for this path (freed in hx_destroy through hx_l2_free).
struct hx_l2_scratch {
    HxDevBuf<int32_t> keys, hist, bstart, perm, chunk_eb, part;
    HxDevBuf<uint8_t> onehot;
};

void hx_l2_free(hx_matrix *h) {
    hx_l2_scratch *s = (hx_l2_scratch *)h->l2_scratch;
    if (!s) return;
    cudaStream_t st = h->stream;
    s->keys.release(st); s->hist.release(st); s->bstart.release(st); s->perm.release(st); s->chunk_eb.release(st);
    s->part.release(st); s->onehot.release(st);
    delete s;
    h->l2_scratch = nullptr;
}

// bytes of one-hot operand scratch the path would need (the caller falls back to the tile kernels above a limit)
int64_t hx_lumma_scratch_bytes(const hx_matrix *h, int64_t n_reads) {
    const L2Geom g = L2Geom::make(h->N, h->W);
    const int64_t max_chunks = (n_reads + 31) / 32 + (n_reads < g.NB ? n_reads : g.NB);
    return max_chunks * g.SP * (int64_t)L2_SLAB;
}

// go: optional device flag; the kernels do nothing when it is zero (a wire-format chunk that failed its checks)
int hx_launch_ingest_lumma(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off, const uint8_t *d_codes,
                           int64_t n_reads, const int *go) {
    if (!h->l2_scratch) h->l2_scratch = new hx_l2_scratch();
    hx_l2_scratch *s = (hx_l2_scratch *)h->l2_scratch;
    cudaStream_t st = h->stream;
    const L2Geom g = L2Geom::make(h->N, h->W);
    const int64_t nbins = g.n_bins();
    const int64_t max_chunks = (n_reads + 31) / 32 + (n_reads < g.NB ? n_reads : g.NB);
    HX_CHECK_ARG(n_reads < ((int64_t)1 << 30) && nbins < ((int64_t)1 << 30));
    constexpr int ITEMS = 16;
    const int64_t nscan = nbins + 1;
    const int64_t nblk = (nscan + 256 * ITEMS - 1) / (256 * ITEMS);
    HX_CUDA(s->keys.grow(sizeof(int32_t) * n_reads, st));
    HX_CUDA(s->hist.grow(sizeof(int32_t) * (2 * nscan + 4), st));         // histogram | cursors | tile counter
    HX_CUDA(s->bstart.grow(sizeof(int32_t) * nscan, st));
    HX_CUDA(s->perm.grow(sizeof(int32_t) * max_chunks * 32, st));
    HX_CUDA(s->chunk_eb.grow(sizeof(int32_t) * max_chunks, st));
    HX_CUDA(s->part.grow(sizeof(int32_t) * nblk, st));
    const int64_t onehot_bytes = max_chunks * g.SP * (int64_t)L2_SLAB;
    HX_CUDA(s->onehot.grow(onehot_bytes + L2P_G * (int64_t)L2_SLAB, st));  // + zero slabs
    int32_t *cursor = s->hist.p + nscan;

    HX_CUDA(hx_fill_async(s->hist.p, 0, sizeof(int32_t) * (size_t)(2 * nscan + 4), st));
    HX_CUDA(hx_fill_async(s->perm.p, 0xff, sizeof(int32_t) * (size_t)(max_chunks * 32), st));
    const unsigned rgrid = (unsigned)((n_reads + 255) / 256);
    k_l2_keys<<<rgrid, 256, 0, st>>>(d_rank, d_off, n_reads, g, s->keys.p, s->hist.p, h->d_err.p, go);
    k_l2_pad<<<(unsigned)((g.NB + 255) / 256), 256, 0, st>>>(s->hist.p, g, go);
    k_scan_partials<int32_t, 0, ITEMS><<<(unsigned)nblk, 256, 0, st>>>(s->hist.p, nscan, s->part.p);
    k_scan_spine<int32_t, 0><<<1, 32, 0, st>>>(s->part.p, nblk, nullptr);
    k_scan_apply<int32_t, 0, ITEMS, true><<<(unsigned)nblk, 256, 0, st>>>(s->hist.p, nscan, s->part.p, s->bstart.p);
    k_l2_scatter<<<rgrid, 256, 0, st>>>(s->keys.p, n_reads, s->bstart.p, cursor, s->perm.p, go);
    k_l2_onehot<<<(unsigned)((max_chunks * 32 + 255) / 256), 256, 0, st>>>(d_rank, d_off, d_codes, s->perm.p, s->bstart.p, g,
                                                                           s->onehot.p, s->chunk_eb.p, hx_cnt_ref(h),
                                                                           h->d_totals.p, h->d_err.p, go);
    k_l2_slabs<<<dim3((unsigned)max_chunks, (unsigned)((g.SP + 7) / 8)), 256, 0, st>>>(d_rank, d_off, d_codes, s->perm.p, s->bstart.p, g,
                                                                                     s->onehot.p, h->d_totals.p, h->d_err.p, go);
    const int sms = ingest_sm_budget(h);
    const bool fused = h->peer_world > 1;
    const bool fresh = !fused && h->use.cnt_fresh;
    static const bool pairs_on = getenv("HX_LUMMA_PAIRS") && !strcmp(getenv("HX_LUMMA_PAIRS"), "1");
    if (!fused && sms >= 2 && pairs_on && g.SP <= 62) {
        // CTA pairs (cta_group::2): one cluster of two per TPC
        uint8_t *zero_slabs = s->onehot.p + onehot_bytes;
        HX_CUDA(hx_fill_async(zero_slabs, 0, L2P_G * (size_t)L2_SLAB, st));
        const size_t smem = (size_t)L2P_STAGES * L2P_STAGE_BYTES + (size_t)L2_EP_WARPS * L2_STG_WORDS * 4 + 1024;
        auto kern = fresh ? k_l2_tiles2<true> : k_l2_tiles2<false>;
        HX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<sms & ~1, L2P_THREADS, smem, st>>>(s->onehot.p, zero_slabs, s->bstart.p, g, hx_cnt_ref(h), h->d_totals.p, go);
        h->use.launches++;
    } else {
        const size_t smem = (size_t)L2_STAGES * L2_STAGE_BYTES + (size_t)L2_EP_WARPS * L2_STG_WORDS * 4 + 1024;
        const auto kern = ingest_kernel_for(h, [&](auto fused_t) {
            constexpr bool F = decltype(fused_t)::value;
            return fresh ? k_l2_tiles<false, true> : k_l2_tiles<F, false>;      // fresh: a single-GPU build only
        });
        HX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<sms, L2_THREADS, smem, st>>>(s->onehot.p, s->bstart.p, g, hx_cnt_ref(h), h->d_totals.p, go);
    }
    h->use.launches += 11;
    HX_CUDA(cudaGetLastError());
    return HX_OK;
}
