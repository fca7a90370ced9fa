// K1 on the 5th-generation tensor cores: pair expansion as an integer rank-k update.
// Replaces gretel/util.py:226-286 (+ Hansel.add_observation) for rank-sorted reads of at most 32 SNPs.
//
// Reads that share a rank r (same first SNP) cover the same sites r+1..r+k.  Write such a read as a one-hot
// row x over the columns (site t, allele a in ACGT): x[4t+a] = 1.  The counts the read adds to every site pair
// (t1 < t2) and allele pair (a, b) are exactly the entries of the outer product x^T x, so a run of reads of one
// rank contributes C = X^T X with X = [reads x columns] in {0,1}.  That is an int8 GEMM with int32 accumulation
// (tcgen05.mma kind::i8: exact by construction), M = N = columns (<= 128), K = reads:
//
//   slices           a CTA takes an equal share of the WEIGHT of the rank-sorted reads (alleles, reads, ranks:
//                    hx_weighted_slice), builds the table of its jobs (one job = up to 32 reads of one run = the K of
//                    one MMA) with a block scan over the runs of its slice, then splits into
//   expander warps   (24) job e, e+24, ...; lane = read: load its allele bytes, turn four sites at a time into four
//                    one-hot words (1 << 8*code; N, -, _ and positions past the read's end give 0) and store them
//                    with one 16-byte shared-memory store into the warp's own operand slot.  The row of a read IS the
//                    MN-major UMMA operand layout (core matrix = 16 columns x 8 reads), so there is no transpose
//                    anywhere.  Lane 0 issues the tcgen05.mma (M=128, N=16*ceil(k/4), K=32; A and B descriptors point
//                    at the same slot) into the run's accumulator stage in TMEM (four stages of 128 columns) and
//                    commits it to the slot's mbarrier and to the stage's completion barrier.
//   readout warps    (8) one run at a time: wait for the stage, tcgen05.ld the upper triangle of C, add it into the
//                    CTA's sliding shared-memory tile of band rows (as k1_bitsliced does), zero the stage, flush
//                    retired rows to HBM with integer reductions.
//
// Reads holding N, - or _, the sentinels and the totals are handled per read by the expander warps exactly as
// in the bit-sliced kernels (ingest_common.cuh).
#include <stdlib.h>

#include <algorithm>

#include "hx_internal.cuh"
#include "ingest_common.cuh"

namespace {

#ifndef UM_EXP_WARPS_N
#define UM_EXP_WARPS_N 24
#endif
constexpr int UM_RD_WARPS = 8;               // readout warps: two per TMEM lane quarter (warp id % 4)
constexpr int UM_EXP_WARPS = UM_EXP_WARPS_N; // expander warps 8..
constexpr int UM_THREADS = (UM_RD_WARPS + UM_EXP_WARPS) * 32;
#ifndef UM_GATE_NS
#define UM_GATE_NS 200
#endif
constexpr int UM_JB = 256;                  // runs per batch of the job-table build
constexpr int UM_NACC = 4;                   // accumulator stages (runs in flight)
constexpr int UM_TMEM_COLS = 128 * UM_NACC;  // 128 int32 columns each
constexpr uint32_t UM_ACC_COUNT = 1u << 19;  // arrivals that complete an accumulator stage (see the readout warps)

#ifdef UM_PROFILE
__device__ unsigned long long um_prof[32];
#define UM_T(var) const long long var = clock64()
#define UM_ACC(slot, expr) prof_acc[slot] += (unsigned long long)(expr)
#else
#define UM_T(var)
#define UM_ACC(slot, expr)
#endif

struct UmLayout {
    int kmax;
    __host__ __device__ int ch() const { return kmax <= 16 ? 4 : 8; }
    __host__ __device__ size_t slot_bytes() const { return (size_t)32 * 16 * ch(); }       // one group of 32 reads
    __host__ __device__ size_t tile_bytes() const { return (size_t)(kmax + 1) * (kmax - 1) * 64; }
    __host__ __device__ size_t bytes() const {
        return (size_t)UM_EXP_WARPS * slot_bytes() + tile_bytes() + 1024;   // tile behind the slots (see um_desc)
    }
};

__device__ __forceinline__ uint32_t um_shl(uint32_t v, uint32_t amt) {      // shl.b32 clamps: amt >= 32 -> 0
    uint32_t r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(amt));
    return r;
}

// Shared-memory matrix descriptor (tcgen05, SWIZZLE_NONE, MN-major): core matrix = 16 contiguous columns (bytes) x
// 8 reads at a 16-byte pitch; the next 16 columns are SBO = 128 bytes away, the next 8 reads LBO bytes away.
__device__ __forceinline__ uint64_t um_desc(uint32_t saddr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fffu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16;
    d |= (uint64_t)((128u >> 4) & 0x3fffu) << 32;
    d |= (uint64_t)1 << 46;                                   // descriptor version (Blackwell)
    return d;                                                 // base offset 0, layout type 0 = no swizzle
}

// Instruction descriptor, kind::i8: unsigned 8-bit A and B (both MN-major), int32 accumulators, M = 128.
__device__ __forceinline__ uint32_t um_idesc(int n_cols) {
    return (2u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(n_cols >> 3) << 17) | ((128u >> 4) << 24);
}

__device__ __forceinline__ void um_mma(uint32_t tmem_d, uint64_t desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %3, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %1, %2, p;\n\t}"
        ::"r"(tmem_d), "l"(desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void um_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void um_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void um_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void um_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ unsigned um_ld_acquire(uint32_t addr) {
    unsigned v;
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void um_st16_zero(uint32_t taddr) {
    const uint32_t z = 0;
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
        ::"r"(taddr), "r"(z)
        : "memory");
}
__device__ __forceinline__ void um_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void um_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// The schedule, walked identically by every warp: the runs of reads that share a rank, as a compact list in rank
// order (k_run_list below: run_rank[j], run_stop[j] = index after the run's last read), clipped to the CTA's slice
// [lo, hi).  The next entry is requested while the current run is being processed.
struct UmWalk {
    const int32_t *run_rank;
    const int64_t *run_stop;
    int64_t hi, cur, p_stop;
    int n_runs, j, p_rank;
    // the current run
    int64_t start, n;
    int r;
    unsigned ri;

    __device__ __forceinline__ void fetch() {
        if (j < n_runs) { p_rank = run_rank[j]; p_stop = run_stop[j]; }
    }
    __device__ __forceinline__ void init(const int32_t *rr, const int64_t *rs, int n_runs_, int64_t lo_, int64_t hi_) {
        run_rank = rr; run_stop = rs; n_runs = n_runs_; hi = hi_; cur = lo_; ri = 0u - 1u; r = 0; start = lo_; n = 0;
        int a = 0, b = n_runs_;                                 // first run that ends behind lo
        while (a < b) {
            const int m = (a + b) >> 1;
            if (run_stop[m] > lo_) b = m; else a = m + 1;
        }
        j = a;
        p_rank = 0; p_stop = 0;
        fetch();
    }
    __device__ __forceinline__ bool next_run() {
        while (cur < hi && j < n_runs) {
            const int64_t stop = p_stop;
            r = p_rank;
            ++j;
            fetch();
            if (stop <= cur) continue;
            const int64_t run_hi = stop < hi ? stop : hi;
            start = cur;
            n = run_hi - cur;
            cur = run_hi;
            ++ri;
            return true;
        }
        cur = hi;                                               // reads with ranks outside [0,N]: flagged by the pre-pass
        return false;
    }
};

// run_end[0..N] (-1 = no reads of that rank) -> the compact run list, in rank order.  One CTA: every thread takes a
// contiguous piece of the ranks, the piece counts are scanned over the block, then the pieces are written in place.
__global__ void __launch_bounds__(1024)
k_run_list(const int64_t *__restrict__ run_end, int N, int32_t *__restrict__ run_rank, int64_t *__restrict__ run_stop,
           int *__restrict__ n_runs) {
    __shared__ int s_warp[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int per = (N + 1 + 1023) / 1024;
    const int i0 = (int)threadIdx.x * per, i1 = min(i0 + per, N + 1);
    int mine = 0;
    for (int i = i0; i < i1; ++i) mine += run_end[i] >= 0;
    int incl = mine;                                           // inclusive scan over the warp, then over the warps
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += v;
        }
        s_warp[lane] = w;                                      // inclusive over the warps
    }
    __syncthreads();
    int pos = incl - mine + (warp ? s_warp[warp - 1] : 0);
    for (int i = i0; i < i1; ++i) {
        const int64_t e = run_end[i];
        if (e >= 0) { run_rank[pos] = i; run_stop[pos] = e; ++pos; }
    }
    if (threadIdx.x == 1023) *n_runs = s_warp[31];
}

// lane = read: the aligned words holding its allele bytes.  The number of words is warp-uniform (what the widest
// read of the group needs at the worst alignment): a narrower read loads a few bytes of its successors, which the
// expansion masks; the packed codes are padded, so the loads stay in bounds.
template <int CH>
__device__ __forceinline__ void um_load_read(const uint8_t *__restrict__ codes, int64_t o, int kg,
                                             uint32_t (&wd)[CH + 1], unsigned &mis) {
    const uint8_t *__restrict__ c = codes + o;
    mis = (unsigned)(reinterpret_cast<uintptr_t>(c) & 3u);
    const uint32_t *__restrict__ cw = reinterpret_cast<const uint32_t *>(c - mis);
    const int nwg = (kg + 6) >> 2;                                  // ceil((3 + kg) / 4) words
#pragma unroll
    for (int w = 0; w <= CH; ++w) wd[w] = w < nwg ? __ldg(cw + w) : 0u;
}

// ... and their expansion into the one-hot operand row (CH chunks of four sites, one 16-byte store each).
template <int CH>
__device__ __forceinline__ void um_expand_read(const uint32_t (&wd)[CH + 1], unsigned mis, int kb, int kg,
                                               uint32_t rowaddr, uint32_t &rare_or, uint32_t &x0) {
    const unsigned sh = 8u * mis;
    const int kb8 = 8 * kb;
    rare_or = 0;
    x0 = 0x04040404u;
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
        uint32_t o0 = 0, o1 = 0, o2 = 0, o3 = 0;
        if (4 * ch < kg) {                                        // warp-uniform
            const uint32_t xx = __funnelshift_r(wd[ch], wd[ch + 1], sh);
            const int c8 = min(max(kb8 - 32 * ch, 0), 32);        // valid bits of this word
            const uint32_t inval = um_shl(0xffffffffu, (uint32_t)c8);   // bytes past the read's end
            rare_or |= xx & 0xfcfcfcfcu & ~inval;
            const uint32_t x = (xx & ~inval) | (0x04040404u & inval);   // past the end -> 'N' -> no column
            if (ch == 0) x0 = x;
            const uint32_t y = x << 3;                            // byte j = 8 * code of site 4ch+j
            o0 = um_shl(1u, __byte_perm(y, 0u, 0x4440u));
            o1 = um_shl(1u, __byte_perm(y, 0u, 0x4441u));
            o2 = um_shl(1u, __byte_perm(y, 0u, 0x4442u));
            o3 = um_shl(1u, y >> 24);
        }
        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(rowaddr + (uint32_t)ch * 128u), "r"(o0), "r"(o1),
                     "r"(o2), "r"(o3)
                     : "memory");
    }
}

template <int CH, bool FUSED>
__global__ void __launch_bounds__(UM_THREADS, 1)
k1_umma(const int32_t *__restrict__ rank, const int64_t *__restrict__ off, const uint8_t *__restrict__ codes,
        int64_t n_reads, int N, int W, int kmax, const HxCnt cnt_in, unsigned long long *__restrict__ totals,
        int *__restrict__ err, const int *__restrict__ sorted_flag, const int32_t *__restrict__ run_rank,
        const int64_t *__restrict__ run_stop, const int *__restrict__ n_runs_ptr, int4 *__restrict__ jobs_all,
        int jobs_cap, int read_w, int rank_w) {
    extern __shared__ __align__(1024) uint8_t um_smem[];
    UM_T(k_begin);
    const HxCnt cnt = cnt_in.for_build<FUSED>();
    __shared__ __align__(8) unsigned long long s_slot[UM_EXP_WARPS];   // a warp's operand slot has been read by its MMA
    __shared__ __align__(8) unsigned long long s_acc_full[UM_NACC];    // all MMAs of a run are complete
    __shared__ int s_runkg[UM_NACC];                       // widest read of the run accumulating in each stage
    __shared__ unsigned s_runs_read;                 // runs read out of TMEM (and their stage zeroed again)
    __shared__ uint32_t s_tmem;
    __shared__ int s_jb_off[UM_JB + 1], s_jb_start[UM_JB], s_jb_n[UM_JB], s_jb_r[UM_JB], s_jb_warp[UM_JB / 32];
    __shared__ int s_njobs;
    if (!*sorted_flag) return;                       // the generic fallback launch takes over

    constexpr int ROWB = 16 * CH;                    // bytes of one read's operand row
    constexpr uint32_t LBO = 128u * CH;              // 8 reads further
    constexpr uint32_t SLOTB = 32u * ROWB;           // one group: 32 reads = the K of one MMA

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t lo, hi;                                  // equal shares of the work, not of the read count
    hx_weighted_slice(rank, off, n_reads, read_w, rank_w, lo, hi);
    if (lo >= hi) return;

    const int rows = kmax + 1, cells = kmax - 1;
    const uint32_t x_saddr = hx_smem_u32(um_smem);
    uint4 *const tile = reinterpret_cast<uint4 *>(um_smem + (size_t)UM_EXP_WARPS * SLOTB);
    uint32_t *const tile32 = reinterpret_cast<uint32_t *>(tile);

    for (size_t w = threadIdx.x; w < (size_t)rows * cells * 4; w += blockDim.x) tile[w] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        s_runs_read = 0;
        for (int s = 0; s < UM_NACC; ++s) s_runkg[s] = 0;
        for (int e = 0; e < UM_EXP_WARPS; ++e) hx_mbar_init(hx_smem_u32(&s_slot[e]), 1);
        for (int s = 0; s < UM_NACC; ++s) hx_mbar_init(hx_smem_u32(&s_acc_full[s]), UM_ACC_COUNT);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(hx_smem_u32(&s_tmem)),
                     "r"((uint32_t)UM_TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    um_fence_before();
    __syncthreads();
    um_fence_after();
    const uint32_t tmem_base = s_tmem;
    if (warp < UM_RD_WARPS) {
        // every MMA accumulates (they are issued by many warps in no particular order): the stages start at zero and
        // the readout warps zero what they have read.  Warps 0-3 clear the even stages, warps 4-7 the odd ones.
        for (int st = warp >> 2; st < UM_NACC; st += 2) {
            const uint32_t t0 = tmem_base + (uint32_t)st * 128u + ((uint32_t)((warp & 3) * 32) << 16);
#pragma unroll
            for (int cb = 0; cb < 128; cb += 16) um_st16_zero(t0 + (uint32_t)cb);
        }
        um_wait_st();
    }
    um_fence_before();
    __syncthreads();
    um_fence_after();

    unsigned long long t_crumbs = 0;
    unsigned n_slices = 0, n_codes = 0, n_notcov = 0, n_sent = 0, n_rcrumbs = 0, errbits = 0;
#ifdef UM_PROFILE
    unsigned long long prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif

    UmWalk wk;
    wk.init(run_rank, run_stop, *n_runs_ptr, lo, hi);

    // ---- the CTA's job table.  A job = one group of up to 32 reads of one run = the K of one MMA, as
    // (first read - lo, reads | run length << 8 on a run's first job, rank, run index).  The runs of the slice are taken
    // UM_JB at a time: a block scan of their group counts gives every run its place, then all threads write the jobs.
    // The expander warps read their jobs from the table instead of each walking the run list.
    int4 *const myjobs = jobs_all + (size_t)blockIdx.x * jobs_cap;
    {
        const int n_runs_all = *n_runs_ptr;
        const int j0 = wk.j;                                   // first run that ends behind lo
        int job_base = 0;
        for (int jb = j0; jb < n_runs_all; jb += UM_JB) {
            int ng = 0;
            if (threadIdx.x < UM_JB) {
                const int j = jb + (int)threadIdx.x;
                int64_t s0 = hi;
                if (j < n_runs_all) {
                    const int64_t prev = j > 0 ? run_stop[j - 1] : 0;
                    s0 = prev > lo ? prev : lo;
                }
                if (s0 < hi) {
                    const int64_t stop = run_stop[j];
                    const int64_t e0 = stop < hi ? stop : hi;
                    ng = (int)((e0 - s0 + 31) >> 5);
                    s_jb_start[threadIdx.x] = (int)(s0 - lo);
                    s_jb_n[threadIdx.x] = (int)(e0 - s0);
                    s_jb_r[threadIdx.x] = run_rank[j];
                }
                int incl = ng;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += v;
                }
                if (lane == 31) s_jb_warp[warp] = incl;
                s_jb_off[threadIdx.x + 1] = incl;              // inclusive within the warp for now
            }
            __syncthreads();
            if (threadIdx.x < UM_JB) {
                int before = 0;
                for (int w2 = 0; w2 < warp; ++w2) before += s_jb_warp[w2];
                const int incl = s_jb_off[threadIdx.x + 1] + before;
                __syncwarp();
                s_jb_off[threadIdx.x + 1] = incl;
                if (threadIdx.x == 0) s_jb_off[0] = 0;
            }
            __syncthreads();
            const int batch_jobs = s_jb_off[UM_JB];
            for (int q = threadIdx.x; q < batch_jobs; q += blockDim.x) {
                int a = 0, b = UM_JB - 1;                      // the run whose jobs hold q: last t with off[t] <= q and off[t+1] > q
                while (a < b) {
                    const int m = (a + b) >> 1;
                    if (s_jb_off[m + 1] > q) b = m; else a = m + 1;
                }
                const int g = q - s_jb_off[a];
                const int n_run = s_jb_n[a];
                const int nj = min(32, n_run - 32 * g);
                myjobs[job_base + q] = make_int4(s_jb_start[a] + 32 * g, nj | (g == 0 ? (min(n_run, 2048) << 8) : 0), s_jb_r[a],
                                                 jb - j0 + a);
            }
            job_base += batch_jobs;
            const bool more = s_jb_off[UM_JB] > s_jb_off[UM_JB - 1];     // the batch's last run was inside the slice
            __syncthreads();
            if (!more) break;
        }
        if (threadIdx.x == 0) s_njobs = job_base;
        __syncthreads();
    }
    UM_T(k_roles);

    if (warp >= UM_RD_WARPS) {
        // ================================ expanders ==========================================
        // A job = one group of 32 reads of a run = the K of one MMA.  Groups are dealt round-robin over the expander
        // warps.  Each warp is a pipeline of its own: request the offsets of its NEXT job, load the alleles of
        // the current one, expand them into its private operand slot, issue the MMA itself and commit it to the
        // slot's mbarrier (slot reusable) and to the run's accumulator barrier (run complete).
        const int e = warp - UM_RD_WARPS;
        const uint32_t slot_addr = x_saddr + (uint32_t)e * SLOTB;
        const uint32_t slot_bar = hx_smem_u32(&s_slot[e]);
        const uint64_t desc = um_desc(slot_addr, LBO);
        const uint32_t idesc0 = um_idesc(0);
        const uint32_t accfull_addr = hx_smem_u32(&s_acc_full[0]);
        const uint32_t rowaddr = slot_addr + (uint32_t)(lane >> 3) * LBO + (uint32_t)(lane & 7) * 16u;
#ifndef UM_PF_READS
#define UM_PF_READS 2048
#endif
        constexpr int64_t PF_READS = UM_PF_READS;               // L2 prefetch distance in reads
        unsigned njobs = 0;
        const int n_jobs = s_njobs;
        // job = (first read - lo, reads | run length << 8 on a run's first job, rank, run index); y = 0: no job left
        auto get_job = [&](int idx) -> int4 {
            int4 j = make_int4(0, 0, 0, 0);
            if (idx < n_jobs) j = myjobs[idx];
            return j;
        };
        auto load_off = [&](const int4 &j, int64_t &o, int64_t &o1) {
            o = 0; o1 = 0;
            if (lane < (j.y & 0xff)) { const int64_t *p = off + lo + j.x + lane; o = p[0]; o1 = p[1]; }
        };
        const uint32_t runs_addr = hx_smem_u32(&s_runs_read);
        int ji = e;
        int4 cur = get_job(ji);
        int64_t o, o1;
        load_off(cur, o, o1);
        while (cur.y) {
            UM_T(tA);
            ji += UM_EXP_WARPS;
            const int4 nxt = get_job(ji);
            int64_t on, o1n;
            load_off(nxt, on, o1n);                             // in flight while this job is expanded
            if (lane == 0 && (cur.y >> 8)) {
                // a run's first job: the packed reads are streamed from HBM exactly once: request the offsets and
                // (extrapolated from this job's byte range) the codes of the reads PF_READS further on
                const int64_t start = lo + cur.x, n_run = cur.y >> 8;
                const int64_t pf0 = start + PF_READS;
                if (pf0 < hi) {
                    const int64_t np = min(n_run, hi - pf0);
                    bs_prefetch_l2(off + pf0, (uint32_t)((np + 1) * 8));
                    const int nj = cur.y & 0xff;
                    const int64_t o_lo = o, o_hi = off[start + nj];
                    const int64_t per_read16 = ((o_hi - o_lo) << 4) / nj;
                    bs_prefetch_l2(codes + o_lo + ((PF_READS * per_read16) >> 4), (uint32_t)(((np * per_read16) >> 4) + 64));
                }
            }
            const int r = cur.z;
            const unsigned cur_ri = (unsigned)cur.w;
            const int s = cur_ri % UM_NACC;
            // SNPs on my read: 0 for a lane past the run's end or a read with fewer than two
            const int64_t kd = o1 - o;
            int kb = 0;
            if ((uint64_t)kd >= 2) {                                // offsets that decrease (kd < 0) are an error too
                if (kd < 0 || !read_fits(r, kd, N, W)) errbits |= 1;
                else kb = (int)kd;
            }
            n_slices += kb >= 2;
            n_codes += kb;
            const int kg = __reduce_max_sync(0xffffffffu, kb);
            UM_T(tC);
            uint32_t wd[CH + 1];
            unsigned mis;
            um_load_read<CH>(codes, o, kg, wd, mis);
            UM_T(tD);
            // the run's accumulator stage: run ri-NACC must have been read out (and the stage zeroed) before anything
            // of run ri is added; the previous MMA of this warp must have read the slot before it is rewritten
            if (cur_ri >= (unsigned)UM_NACC) {
                const unsigned need = cur_ri - UM_NACC + 1;
                while (um_ld_acquire(runs_addr) < need) __nanosleep(UM_GATE_NS);
            }
            hx_mbar_wait(slot_bar, (njobs & 1) ^ 1);
            um_fence_after();
            UM_T(tE);
            uint32_t rare_or, x0;
            um_expand_read<CH>(wd, mis, kb, kg, rowaddr, rare_or, x0);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic stores -> tensor-core reads
            __syncwarp();
            if (lane == 0) {
                if (kg >= 2) {
                    const int c4 = (kg + 3) >> 2;                   // chunks of four sites the group reaches
                    atomicMax(&s_runkg[s], kg);
                    asm volatile("fence.acq_rel.cta;" ::: "memory");
                    um_mma(tmem_base + (uint32_t)s * 128u, desc, idesc0 | ((uint32_t)c4 << 18), 1u);
                }
                um_commit(slot_bar);
                um_commit(accfull_addr + 8u * (uint32_t)s);
            }
            ++njobs;
            UM_T(tG);
            if (r == 0 || r + kg >= N) {                            // warp-uniform: runs at the ends of the region
                if (kb >= 2) add_sentinels(codes + o, x0 & 0xffu, r, kb, N, W, cnt, n_sent);
            }
            // reads holding N, - or _: their pairs with such an allele are added right here by the warp
            unsigned rm = __ballot_sync(0xffffffffu, kb >= 2 && rare_or != 0);
            while (rm) {
                const int src = __ffs(rm) - 1;
                rm &= rm - 1;
                const int64_t o2 = __shfl_sync(0xffffffffu, o, src);
                const int k2 = __shfl_sync(0xffffffffu, kb, src);
                bs_rare_read<false>(codes + o2, k2, r, W, cnt, n_rcrumbs, n_notcov, errbits);
            }
            UM_T(tH);
            UM_ACC(0, tC - tA); UM_ACC(1, tD - tC); UM_ACC(2, tE - tD); UM_ACC(3, tG - tE); UM_ACC(4, tH - tG); UM_ACC(5, 1);
            cur = nxt; o = on; o1 = o1n;
        }
#ifdef UM_PROFILE
        if (lane == 0) for (int i = 0; i < 6; ++i) atomicAdd(&um_prof[i], prof_acc[i]);
#endif
    } else {
        // ================================ readout ============================================
        // 8 warps: warp w reads TMEM lanes 32*(w%4).. (rows = (site t1, allele a) of the run) and every other block of
        // 16 columns (= 4 sites t2); only t2 > t1 is a site pair.
        const int npt = UM_RD_WARPS * 32;
        const int q = warp & 3, half = warp >> 2;
        const int m = q * 32 + lane, t1 = m >> 2, a = m & 3;
        const int per_row = cells * 16;
        // where this thread's tile words (tid and tid + 256 of a row of cells x 16 counters) live in a band row
        auto word_off = [](int w) { return (w >> 4) * HX_CELL + ((w & 15) >> 2) * HX_NSYM + (w & 3); };
        const int goff0 = word_off(threadIdx.x), goff1 = word_off(threadIdx.x + npt);
        static_assert(UM_RD_WARPS * 32 * 2 >= 31 * 16, "two tile words per readout thread cover a band row");
        int64_t flushed_upto = (int64_t)max(rank[lo], 0) + 1;  // (a negative rank is an error the pre-pass has flagged)
        while (wk.next_run()) {
            const int r = wk.r;
            const unsigned ri = wk.ri;
            const int s = ri % UM_NACC;
            UM_T(r0);
            // (the tile adds of the previous run are complete: barrier at the end of the loop body)
            if ((int64_t)r + 1 > flushed_upto) {
                // the rows flushed below and the rows this run adds to (r+2 .. r+kmax) share a ring slot only if the
                // ranks jumped: rows of the ring are kmax+1 apart
                const bool slots_reused = (int64_t)r - flushed_upto >= 2;
                const int64_t lastrow = min((int64_t)r + 1, flushed_upto + rows - 2);
                // rows pj <= r+1 can no longer be touched by this CTA
                unsigned long long sum = 0;
                int row = (int)((unsigned)(flushed_upto + 1) % (unsigned)rows);
                for (int64_t pj = flushed_upto + 1; pj <= lastrow; ++pj) {
                    uint32_t *base = tile32 + (size_t)row * per_row;
                    uint32_t *grow = cnt.cell(W, pj - 1, pj);        // cell d = 1 of band row pj; cell d is 49*(d-1) further
                    for (int w = threadIdx.x, k2 = 0; w < per_row; w += npt, ++k2) {
                        const uint32_t v = base[w];
                        if (v) {
                            atomicAdd(grow + (k2 ? goff1 : goff0), v);
                            base[w] = 0;
                            sum += v;
                        }
                    }
                    if (++row == rows) row = 0;
                }
                t_crumbs += sum;
                flushed_upto = (int64_t)r + 1;
                if (slots_reused) ws_pair_barrier(npt);   // retired ring slots are reused by this run's tile add
            }
            const int rbase = (int)((unsigned)(r + 1) % (unsigned)rows);
            UM_T(r1);
            // the stage is complete after UM_ACC_COUNT arrivals: one per group (the expanders' commits) plus the rest here
            if (threadIdx.x == 0) {
                const uint32_t ng = (uint32_t)((wk.n + 31) >> 5);
                asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0], %1;" ::"r"(hx_smem_u32(&s_acc_full[s])),
                             "r"(UM_ACC_COUNT - ng)
                             : "memory");
            }
            hx_mbar_wait(hx_smem_u32(&s_acc_full[s]), (ri / UM_NACC) & 1);
            um_fence_after();
            UM_T(r2);
            const int kg = *reinterpret_cast<volatile int *>(&s_runkg[s]);
            const int ncols = 4 * kg;
            const uint32_t taddr = tmem_base + (uint32_t)s * 128u + ((uint32_t)(q * 32) << 16);
            if (kg >= 2) {
                if (q * 32 < ncols - 4) {                                // this lane quarter holds live rows
                    for (int cb = q * 32 + 16 * half; cb < ncols; cb += 32) {
                        uint32_t v[16];
                        um_ld16(taddr + (uint32_t)cb, v);
                        um_wait_ld();
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int t2 = (cb >> 2) + j;
                            if (t2 > t1 && t2 < kg) {
                                int row = rbase + t2;
                                if (row >= rows) row -= rows;
                                uint4 *cell = tile + ((size_t)row * cells + (t2 - t1 - 1)) * 4 + a;
                                uint4 c = *cell;
                                c.x += v[4 * j + 0]; c.y += v[4 * j + 1]; c.z += v[4 * j + 2]; c.w += v[4 * j + 3];
                                *cell = c;
                            }
                        }
                    }
                }
                // zero everything the run's MMAs may have written (all rows, the lower triangle too)
                const int ncols16 = 16 * ((kg + 3) >> 2);
                for (int cb = 16 * half; cb < ncols16; cb += 32) um_st16_zero(taddr + (uint32_t)cb);
                um_wait_st();
            }
            um_fence_before();
            ws_pair_barrier(npt);                // tile adds and zeroing done
            if (threadIdx.x == 0) {
                s_runkg[s] = 0;
                asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(hx_smem_u32(&s_runs_read)), "r"(ri + 1) : "memory");
            }
            UM_T(r3);
            UM_ACC(0, r1 - r0); UM_ACC(1, r2 - r1); UM_ACC(2, r3 - r2); UM_ACC(3, 1);
        }
        t_crumbs += bs_flush_rows(tile32, rows, cells, flushed_upto + 1, flushed_upto + rows - 1, W, cnt, npt, false);
#ifdef UM_PROFILE
        if (threadIdx.x == 0) for (int i = 0; i < 4; ++i) atomicAdd(&um_prof[16 + i], prof_acc[i]);
#endif
    }
    UM_T(k_roles_end);
    if (errbits) atomicOr(err, (int)errbits);
    um_fence_before();
    flush_totals(n_slices, t_crumbs + n_rcrumbs, (unsigned long long)n_codes - n_notcov, n_sent, totals);   // barriers inside
#ifdef UM_PROFILE
    {
        const long long k_end = clock64();
        if (lane == 0) {
            atomicAdd(&um_prof[24], (unsigned long long)(k_roles - k_begin));
            atomicAdd(&um_prof[25], (unsigned long long)(k_roles_end - k_roles));
            atomicAdd(&um_prof[26], (unsigned long long)(k_end - k_roles_end));
            atomicMax(&um_prof[27], (unsigned long long)(k_end - k_begin));
            if (warp >= UM_RD_WARPS) atomicMax(&um_prof[28], (unsigned long long)(k_roles_end - k_roles));
            else atomicMax(&um_prof[29], (unsigned long long)(k_roles_end - k_roles));
        }
    }
#endif
    if (warp == 0) {
        um_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)UM_TMEM_COLS)
                     : "memory");
    }
}

}  // namespace

#ifdef UM_PROFILE
extern "C" int hx_debug_um_prof(unsigned long long *out, int reset) {
    if (cudaMemcpyFromSymbol(out, um_prof, sizeof(unsigned long long) * 32) != cudaSuccess) return -1;
    if (reset) {
        unsigned long long z[32] = {0};
        cudaMemcpyToSymbol(um_prof, z, sizeof(z));
    }
    return 0;
}
#endif

bool hx_umma_possible(const hx_matrix *h) {
    const int kmax = h->W + 1;
    return kmax >= 2 && kmax <= 32;
}

// rank-sorted reads of at most 32 SNPs; run_end must hold -1 for ranks without reads (hx_launch_ingest fills it)
int hx_launch_ingest_umma(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off, const uint8_t *d_codes,
                          int64_t n_reads, const int64_t *run_end, const int *sorted_flag) {
    const int kmax = h->W + 1;
    const size_t smem = UmLayout{kmax}.bytes();
    const auto kern = ingest_kernel_for(h, [&](auto fused_t) {
        constexpr bool F = decltype(fused_t)::value;
        return kmax <= 16 ? k1_umma<4, F> : k1_umma<8, F>;
    });
    unsigned grid;
    if (int rc = ingest_grid(kern, ingest_sm_budget(h), UM_THREADS, smem, false, n_reads, &grid)) return rc;
    int32_t *run_rank = reinterpret_cast<int32_t *>(h->d_run_list.p);
    int64_t *run_stop = reinterpret_cast<int64_t *>(h->d_run_list.p) + (((size_t)h->N + 2 + 1) / 2);
    int *n_runs = reinterpret_cast<int *>(run_stop + (size_t)h->N + 2);
    k_run_list<<<1, 1024, 0, h->stream>>>(run_end, h->N, run_rank, run_stop, n_runs);
    h->use.launches++;
    // slices hold equal shares of (alleles + read_w * reads + rank_w * ranks spanned) - the per-allele, per-read and
    // per-run costs of the kernel (config 3, tuned on the B200: 16 / 8192 gives 0.330 ms per step, equal read counts
    // 0.373); a read carries at most kmax alleles, so a slice holds at most (kmax + read_w) / read_w times its even
    // share of the reads (plus the rank term's share)
    static const int read_w = [] { const char *e = getenv("HX_UM_READ_W"); const int v = e ? atoi(e) : HX_SLICE_READ_W; return v < 1 ? 1 : v; }();
    static const int rank_w = [] { const char *e = getenv("HX_UM_RANK_W"); const int v = e ? atoi(e) : HX_SLICE_RANK_W; return v < 0 ? 0 : v; }();
    // per-CTA job tables: a slice of `per` reads holds at most per/32 full groups plus one partial group per run.  No
    // slice holds more than all the reads: where the rank term dominates (few CTAs, many sites, a large rank_w) the
    // weight bound alone reaches hundreds of GB of tables
    const int64_t per_w = (((n_reads + grid - 1) / grid + 1) * (kmax + read_w) + ((int64_t)rank_w * (h->N + 2) + grid - 1) / grid) / read_w + 2;
    const int64_t per = std::min(per_w, n_reads);
    const int64_t jobs_cap = per / 32 + std::min<int64_t>((int64_t)h->N + 2, per) + 2;
    HX_CHECK_ARG(jobs_cap < ((int64_t)1 << 31) && per < ((int64_t)1 << 31));
    const int64_t jobs_bytes = jobs_cap * grid * (int64_t)sizeof(int4);
    if (jobs_bytes > h->d_jobs.cap) HX_CUDA(h->d_jobs.grow(jobs_bytes + jobs_bytes / 8, h->stream));   // with headroom
    kern<<<grid, UM_THREADS, smem, h->stream>>>(d_rank, d_off, d_codes, n_reads, h->N, h->W, kmax, hx_cnt_ref(h),
                                                h->d_totals.p, h->d_err.p, sorted_flag, run_rank, run_stop, n_runs,
                                                h->d_jobs.p, (int)jobs_cap, read_w, rank_w);
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    return HX_OK;
}
