// K2-K4: haplotype path recovery over the banded Hansel matrix, kept resident on the
// device for the whole walk (no host round trip per site).
//
// Replaces, for the reference (paths under /root/reference):
//   k_site_counts      Hansel.get_counts_at for every site   (cmd.py:85-92,123-145)
//   k_walk_terms/_logm/_tables   gretel.py:143-187 + Hansel.get_edge_weights_at (call gretel.py:155)
//   k_path_stats/_sum  gretel.py:182-189 + Hansel.get_marginal_of_at  (calls :182,186)
//   k_reweight_path    gretel.py:79-98 + Hansel.reweight_observation  (calls :84,96)
//
// All probability arithmetic is float64 on float32-stored cells, in the same
// operation order as oracle/hansel_oracle.c, compiled with -fmad=false so that +,-,*,/
// round exactly like the CPU; log10 and 10**x are evaluated exactly as glibc does (glibc_math.cuh).
#include <limits.h>
#include <stddef.h>
#include <stdlib.h>
#include <math.h>

#include "hx_internal.cuh"
#include "glibc_math.cuh"
#include "recover_common.cuh"

namespace {

// ---- per-site counts -----------------------------------------------------------------
__global__ void k_site_counts(const float *__restrict__ band, int N, int W,
                              double *__restrict__ scnt, int32_t *__restrict__ vseen) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p > N) return;
    const float *cell = band + hx_cell_off(W, p, p + 1);
    double tot = 0.0;
    int v = 0;
    for (int s = 0; s < HX_NSYM; ++s) {
        double c = 0.0;
        for (int b = 0; b < HX_NSYM; ++b) c += (double)cell[s * HX_NSYM + b];
        const bool pos = c > 0;
        scnt[(int64_t)p * 8 + s] = pos ? c : 0.0;
        if (pos) {
            tot += c;
            if (s != HX_SYM_N && s != HX_SYM_GAP) v++;
        }
    }
    scnt[(int64_t)p * 8 + 7] = tot;
    vseen[p] = v;
}

__global__ void __launch_bounds__(32)
k_edge_one(const float *__restrict__ band, const double *__restrict__ scnt,
           const int32_t *__restrict__ vseen, int W, int L, int flags, int snp,
           const uint8_t *__restrict__ path, double *__restrict__ out /* [7] w, [7] total, [8] mask */) {
    unsigned cmask;
    const double ws = edge_weight_lane(band, scnt, vseen, W, L, flags, snp, path, &cmask);
    double wn, tw;
    (void)normalise_and_pick(ws, cmask, &wn, &tw);
    const int lane = threadIdx.x;
    if (lane < HX_NSYM) out[lane] = ((cmask >> lane) & 1u) ? wn : 0.0;
    if (lane == 0) { out[7] = tw; out[8] = (double)cmask; }
}

// ---- staged walk tables ------------------------------------------------------------------------------------------
// Three shared-memory buffers that TMA bulk copies fill with the walk tables of up to C consecutive sites each: first
// the terms of all three buffers ([C][rows][7][8] T each), then their log-marginal rows ([C][8] T each); one mbarrier
// per buffer.  Chunk k of a range holds sites first + kC, ...  A CTA may stage several ranges through the same buffers
// (walk_q_range), so chunk k is the CTA's use number use0 + k: its buffer is that modulo 3, its phase that / 3, mod 2.
template <class T>
struct TableRing {
    static constexpr uint32_t ROW = 8 * sizeof(T);          // bytes of one log-marginal row
    const T *terms, *logm;                                   // global tables: rows*56 and 8 T per site
    uint32_t sm, bars;                                       // shared addresses of buffer 0 and mbarrier 0
    uint32_t site_bytes, chunk_bytes;                        // terms of one site, of one buffer
    int rows, C, first, last, nchunks;
    uint32_t use0;

    // lane 0, once per CTA before any use
    __device__ static void init(unsigned long long *bars) {
        for (int b = 0; b < 3; ++b) hx_mbar_init(hx_smem_u32(&bars[b]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __device__ TableRing(const T *terms_, const T *logm_, int rows_, int C_, int first_, int last_, void *smem,
                         unsigned long long *bars_, uint32_t use0_)
        : terms(terms_), logm(logm_), sm(hx_smem_u32(smem)), bars(hx_smem_u32(bars_)),
          site_bytes((uint32_t)rows_ * 56u * (uint32_t)sizeof(T)), chunk_bytes((uint32_t)C_ * site_bytes), rows(rows_),
          C(C_), first(first_), last(last_), nchunks((last_ - first_ + 1 + C_ - 1) / C_), use0(use0_) {}
    __device__ int buf(int k) const { return (int)((use0 + (uint32_t)k) % 3u); }
    __device__ uint32_t terms_at(int k) const { return sm + (uint32_t)buf(k) * chunk_bytes; }
    __device__ uint32_t logm_at(int k) const { return sm + 3u * chunk_bytes + (uint32_t)buf(k) * C * ROW; }
    // lane 0: stage chunk k into its buffer (nothing past the last chunk)
    __device__ void issue(int k) const {
        if (k >= nchunks) return;
        const int s0 = first + k * C;
        const int ns = min(C, last - s0 + 1);
        const uint32_t bar = bars + 8u * (uint32_t)buf(k);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // earlier reads of this buffer are done
        hx_mbar_expect_tx(bar, (uint32_t)ns * (site_bytes + ROW));
        hx_bulk_g2s(terms_at(k), terms + (int64_t)s0 * rows * 56, (uint32_t)ns * site_bytes, bar);
        hx_bulk_g2s(logm_at(k), logm + (int64_t)s0 * 8, (uint32_t)ns * ROW, bar);
    }
    __device__ void wait(int k) const {
        hx_mbar_wait(bars + 8u * (uint32_t)buf(k), ((use0 + (uint32_t)k) / 3u) & 1u);
    }
    // before a CTA leaves early at chunk k: the copies still in flight must land before its shared memory is released
    __device__ void drain_after(int k) const {
        for (int k2 = k + 1; k2 <= k + 2 && k2 < nchunks; ++k2) wait(k2);
    }
};

// The pick at one site of the float64 walks: lane = candidate symbol, every lane of the warp calls it.  `lwf` is the
// lane's log weight summed in any order.  The reference's ordered sum, 10**x and normalisation
// (Hansel.get_edge_weights_at) only matter for the argmax when two candidates are within rounding of each other, so
// they are evaluated only then (and whenever 10**x could under/overflow); otherwise the largest log weight wins
// outright.  The exact evaluation reads the log-marginal row `lmrow`, the site's terms `tab` ([lt][7][8]) and the
// chosen symbols in `ring`.  CAND_ONLY keeps the other lanes out of it: faster where `tab` is in global memory
// (k_walk_wide), slower where it is in shared memory (k_walk_tables), measured on a B200.  Returns the symbol, or -1
// for a site without a candidate (gretel.py:176-180).
template <bool CAND_ONLY>
__device__ __forceinline__ int pick_site(double lwf, unsigned cmask, const double *lmrow, const double *tab,
                                         const uint8_t *ring, int snp, int lt, int lmax,
                                         const int32_t *__restrict__ vseen, int flags) {
    const int lane = threadIdx.x & 31;
    const bool cand = lane < HX_NSYM && ((cmask >> lane) & 1u);
    // best log weight over the 7 candidate lanes (butterfly), then who is within 1e-6 of it
    const double key = cand ? lwf : -INFINITY;
    double best = key;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) best = fmax(best, __shfl_xor_sync(0xffffffffu, best, o));
    best = __shfl_sync(0xffffffffu, best, 0);    // lanes 8..31 hold -inf: make the branch below warp-uniform
    const unsigned near = __ballot_sync(0xffffffffu, cand && key >= best - 1e-6);
    if (cmask == 0) return -1;
    if (__popc(near) == 1 && best > -300.0 && best < 300.0) return __ffs(near) - 1;   // a clear winner
    // exact evaluation in the reference's order: ((log10 P(s) + t1) + t2) + ...
    const int s = CAND_ONLY || lane < HX_NSYM ? lane : 0;     // lanes 7..31 repeat symbol 0's sums, which are not used
    double lw = 0.0;
    if (!CAND_ONLY || cand) {
        lw = lmrow[s];
        for (int l = 1; l <= lt; ++l) lw += tab[((l - 1) * HX_NSYM + ring[(snp - l) & (HX_RING - 1)]) * 8 + s];
        lw = add_beyond_band(lw, vseen, flags, snp, lt + 1, lmax);
    }
    const double ws = cand ? hx_gl_pow10(lw) : 0.0;
    double wn, tw;
    return normalise_and_pick(ws, cmask, &wn, &tw);
}

// The walk over the precomputed tables: one warp, lanes 0..6 = candidate symbols, strictly
// sequential over sites.  The tables of the next sites are staged into shared memory (TableRing, three chunks of C
// sites in flight), so the dependent chain per site is: previous choice -> one shared-memory load -> one add ->
// 7-way argmax (pick_site).
__global__ void __launch_bounds__(32)
k_walk_tables(const double *__restrict__ terms, const double *__restrict__ logm,
              const int32_t *__restrict__ vseen, int N, int L, int Lw, int flags, int C,
              uint8_t *__restrict__ path, hx_dev_flags *__restrict__ df) {
    extern __shared__ __align__(128) unsigned char smraw[];
    __shared__ __align__(8) unsigned long long bars[3];
    __shared__ uint8_t ring[HX_RING];
    const int lane = threadIdx.x;
    const int s = lane < HX_NSYM ? lane : 0;
    if (df->hole) return;
    const TableRing<double> tr(terms, logm, Lw, C, 1, N, smraw, bars, 0);
    const double *const sm_terms = reinterpret_cast<const double *>(smraw);                        // [3][C][Lw][7][8]
    const double *const sm_logm = sm_terms + 3 * (size_t)(tr.chunk_bytes / 8);                      // [3][C][8]
    if (lane == 0) {
        ring[0] = HX_SYM_GAP;
        path[0] = HX_SYM_GAP;
        TableRing<double>::init(bars);
    }
    __syncwarp();
    if (lane == 0) { tr.issue(0); tr.issue(1); }
    unsigned last = HX_SYM_GAP;
    unsigned long long hist = HX_SYM_GAP;               // 4 bits per chosen symbol, newest in bits 0..3
    for (int k = 0; k < tr.nchunks; ++k) {
        __syncwarp();
        if (lane == 0) tr.issue(k + 2);
        tr.wait(k);
        const int first = 1 + k * C;
        const int ns = min(C, N - first + 1);
        const double *ct = sm_terms + (size_t)tr.buf(k) * (tr.chunk_bytes / 8);
        const double *cl = sm_logm + (size_t)tr.buf(k) * C * 8;
        for (int j = 0; j < ns; ++j) {
            const int snp = first + j;
            const double *tab = ct + (size_t)j * Lw * 56;
            const double *base = tab + s;
            const double lm = cl[j * 8 + s];
            const unsigned cmask = (unsigned)cl[j * 8 + 7];
            const int lmax = L < snp ? L : snp;
            const int lt = lmax < Lw ? lmax : Lw;
            // the only load that depends on the previous choice
            const double v1 = lt >= 1 ? base[last * 8] : 0.0;
            // everything else, in any order (two accumulators); pick_site restores exactness if needed
            double p0 = lm, p1 = 0.0;
            {
                const int n16 = lt < 16 ? lt : 16;
#pragma unroll
                for (int l = 2; l <= 16; ++l) {
                    if (l <= n16) {
                        const unsigned a = (unsigned)(hist >> (4 * (l - 1))) & 7u;
                        const double v = base[((l - 1) * HX_NSYM + a) * 8];
                        if (l & 1) p1 += v; else p0 += v;
                    }
                }
                for (int l = 17; l <= lt; ++l) {
                    const unsigned a = ring[(snp - l) & (HX_RING - 1)];
                    const double v = base[((l - 1) * HX_NSYM + a) * 8];
                    if (l & 1) p1 += v; else p0 += v;
                }
            }
            const double lwf = (p0 + p1) + add_beyond_band(0.0, vseen, flags, snp, lt + 1, lmax) + v1;
            const int next = pick_site<false>(lwf, cmask, cl + j * 8, tab, ring, snp, lt, lmax, vseen, flags);
            if (next < 0) {                              // gretel.py:176-180
                if (lane == 0) { df->hole_site = snp; df->hole = 1; }
                tr.drain_after(k);
                return;
            }
            last = (unsigned)next;
            hist = (hist << 4) | (unsigned long long)next;
            if (lane == 0) { ring[snp & (HX_RING - 1)] = (uint8_t)next; path[snp] = (uint8_t)next; }
            __syncwarp();
        }
    }
    if (lane == 0) df->hole_site = 0;
}

__device__ __forceinline__ int lds32(uint32_t addr) {
    int v;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// The walk over sites [s_begin, s_end] given the symbols chosen before s_begin (hsrc[site]; site 0 = '_').  One warp.
// Decided symbols go to out[snp - s_begin].  Returns 0, or the site without a candidate (gretel.py:176-180).
template <int NIT>
__device__ __forceinline__ int walk_q_range(const int32_t *__restrict__ termsq, const int32_t *__restrict__ logmq,
                                            const double *__restrict__ terms, const double *__restrict__ logm,
                                            int L, int C, int s_begin, int s_end, const uint8_t *hsrc,
                                            uint8_t *out, bool force_exact, unsigned char *smraw,
                                            unsigned long long *bars, uint32_t &bar_uses) {
    constexpr int Lq = 4 * NIT + 1;
    constexpr uint32_t site_t_bytes = (uint32_t)Lq * 224u;             // int32 terms of one site
    const int lane = threadIdx.x & 31;
    const TableRing<int32_t> tr(termsq, logmq, Lq, C, s_begin, s_end, smraw, bars, bar_uses);
    const int nchunks = tr.nchunks;
    __syncwarp();
    if (lane == 0) { tr.issue(0); tr.issue(1); }
    bar_uses += (uint32_t)nchunks;
    const uint32_t q4 = 4u * (uint32_t)(lane & 7);
    const uint32_t g = (uint32_t)lane >> 3;
    const uint32_t look_off = (1u + g) * 224u + q4;         // this lane's first look-ahead row, its candidate slot
    const uint32_t psel = 0x4440u | g;                      // PRMT selector: byte g of a history word
    // history relative to s_begin - 1: h[t] byte b = 32 * symbol at site (s_begin - 1) - (4t + b + 1); 0 before the start
    uint32_t h[NIT + 1];
#pragma unroll
    for (int t = 0; t <= NIT; ++t) {
        uint32_t w = 0;
#pragma unroll
        for (int bb = 0; bb < 4; ++bb) {
            const int site = s_begin - 1 - (4 * t + bb + 1);
            const uint32_t sym = site >= 0 ? (uint32_t)hsrc[site] : 0u;
            w |= (sym << 5) << (8 * bb);
        }
        h[t] = w;
    }
    unsigned mine = 0;                                      // lane's slot of the 32-site output block
    const int margin_q = 168;                               // 1.6e-4 * 2^20
    // 10**x must stay representable: outside (-300, 300) the exact evaluation decides, where a weight that underflows
    // to 0 or overflows to inf (a lookback term is positive when V = 0 and the support is below 1) changes the
    // normalised weights and so the first-max pick
    const int floor_q = -300 * 1048576, ceil_q = 300 * 1048576;
    tr.wait(0);
    // lookback >= 2 terms of the first site (rows past the start of the region are zero), then its log marginal
    int R;
    {
        const uint32_t site0 = tr.terms_at(0);
        int acc = 0;
#pragma unroll
        for (int t = 0; t < NIT; ++t)
            acc += lds32(site0 + look_off + (uint32_t)t * 896u + __byte_perm(h[t], 0u, psel));
        acc += __shfl_xor_sync(0xffffffffu, acc, 8);
        acc += __shfl_xor_sync(0xffffffffu, acc, 16);
        R = acc + lds32(tr.logm_at(0) + q4);
    }
    // ... and the history relative to s_begin: shift in the symbol at s_begin - 1
    uint32_t prev32 = (uint32_t)hsrc[s_begin - 1] << 5;
#pragma unroll
    for (int t = NIT; t >= 1; --t) h[t] = __funnelshift_l(h[t - 1], h[t], 8);
    h[0] = (h[0] << 8) | prev32;
    for (int k = 0; k < nchunks; ++k) {
        __syncwarp();
        if (lane == 0) tr.issue(k + 2);
        if (k + 1 < nchunks) tr.wait(k + 1);
        const int first = s_begin + k * C;
        const int ns = min(C, s_end - first + 1);
        const uint32_t ct_n = tr.terms_at(k + 1);
        const uint32_t cl_n = tr.logm_at(k + 1);
        uint32_t csite = tr.terms_at(k);                 // current site's table
        uint32_t clm = tr.logm_at(k);
        for (int j = 0; j < ns; ++j) {
            const int snp = first + j;
            // ---- look ahead: lookback >= 2 terms of site snp+1 (independent of this site's choice).  After the
            // last site this reads the next buffer's stale bytes; the result is never used.
            const bool wrap = j + 1 == ns;
            const uint32_t nsite = wrap ? ct_n : csite + site_t_bytes;
            const uint32_t nlm = wrap ? cl_n : clm + 32u;
            int acc = 0;
#pragma unroll
            for (int t = 0; t < NIT; ++t)
                acc += lds32(nsite + look_off + (uint32_t)t * 896u + __byte_perm(h[t], 0u, psel));
            acc += __shfl_xor_sync(0xffffffffu, acc, 8);
            acc += __shfl_xor_sync(0xffffffffu, acc, 16);
            const int Rn = acc + lds32(nlm + q4);
            // ---- the serial chain: lookback-1 term of this site for the symbol just chosen
            const int tot = R + lds32(csite + q4 + prev32);
            const int best = __reduce_max_sync(0xffffffffu, tot);
            const unsigned near = __ballot_sync(0xffffffffu, tot >= best - margin_q) & 0xffu;
            int next = 31 - __clz(near);                     // == ffs-1 when exactly one candidate is near
            if ((near & (near - 1)) != 0 || best <= floor_q || best >= ceil_q || force_exact) {
                const unsigned cmask = (unsigned)logm[(int64_t)snp * 8 + 7];
                if (cmask == 0) next = -1;
                else {
                    // exact evaluation from the float64 tables in the reference's order (lane = candidate)
                    const int lmax = L < snp ? L : snp;
                    const int sy = lane < HX_NSYM ? lane : 0;
                    const bool cand = lane < HX_NSYM && ((cmask >> lane) & 1u);
                    const double *base = terms + ((int64_t)snp * L) * 56 + sy;
                    double lw = logm[(int64_t)snp * 8 + sy];
#pragma unroll
                    for (int l = 1; l <= 4 * NIT + 1; ++l) {
                        if (l <= lmax) {
                            const unsigned al = (h[(l - 1) >> 2] >> (8 * ((l - 1) & 3) + 5)) & 7u;
                            lw += base[((l - 1) * HX_NSYM + al) * 8];
                        }
                    }
                    const double ws = cand ? hx_gl_pow10(lw) : 0.0;
                    double wn, tw;
                    next = normalise_and_pick(ws, cmask, &wn, &tw);
                }
                if (next < 0) {                          // gretel.py:176-180
                    tr.drain_after(k);
                    return snp;
                }
            }
            prev32 = (uint32_t)next << 5;
#pragma unroll
            for (int t = NIT; t >= 1; --t) h[t] = __funnelshift_l(h[t - 1], h[t], 8);
            h[0] = (h[0] << 8) | prev32;
            const int rel = snp - s_begin;
            mine = lane == (rel & 31) ? (unsigned)next : mine;
            if ((rel & 31) == 31 || snp == s_end) {      // a block of 32 sites (or the tail) is complete
                const int at = (rel & ~31) + lane;
                if (at <= rel) out[at] = (uint8_t)mine;
            }
            R = Rn;
            csite = nsite;
            clm = nlm;
        }
    }
    __syncwarp();
    return 0;
}

// Quantised walk (L <= 32, all lookbacks inside the band).  The log terms are kept as 2^-20 fixed point, so a
// candidate's log weight is an exact integer sum in any order.  Lane = (lookback group g = lane/8, candidate
// q = lane%8).  Only the lookback-1 term depends on the symbol chosen at the previous site, so the walk is
// software-pipelined: while site s is being decided, every lane already sums the lookback >= 2 terms of site
// s+1 for its (g,q) (their history is known; rows 1+g, 5+g, ... of the table, NIT per lane) and two shuffles fold
// the four groups.  The serial chain per site is one shared-memory load, an add, a warp max (REDUX), a ballot
// and a find-first-set.  A candidate wins outright only if it leads by more than 1.6e-4 in log10 weight (ten
// times the worst-case quantisation error of 33 terms); otherwise - and whenever 10**x could under/overflow,
// or a term did not fit the fixed-point range - the site is re-evaluated exactly, in the reference's order,
// from the float64 tables (gretel.py:166-174 semantics, first max wins a tie).
// History: h[t] byte b = 32 * symbol chosen 4t+b+1 sites back (byte granular so one PRMT yields a row offset).
//
// PARALLEL IN TIME.  The greedy walk is a chain over sites, but a site only sees the L symbols before it.  So the
// region is cut into blocks that are walked CONCURRENTLY (one CTA each): block b starts `warm` sites early from a
// guessed history (the per-site majority allele) and is SPECULATIVE; k_walk_fix then goes through the blocks in
// order and accepts a block iff the L symbols it chose right before its first site equal the final path there -
// from that point on its choices are exactly what the sequential walk would have made.  A block that fails the
// test (or ran into a site without a candidate) is walked again from the final path.  The result is always the
// sequential greedy walk's; only the time differs (all blocks accepted: N/B + warm sites instead of N).
constexpr int HX_WALK_CAND = 6;      // speculative starts per block: the majority-allele guess + 5 earlier haplotypes

// Which earlier haplotypes a block starts from: the most recent ones whose L symbols before the block differ from
// each other (many of the haplotypes found so far coincide around any one block).  One warp per block.
__global__ void __launch_bounds__(32)
k_walk_pick(const uint8_t *__restrict__ paths0, int it, int N, int L, int blk_len, int *__restrict__ cand_idx) {
    const int b = blockIdx.x, lane = threadIdx.x;
    const int start = 1 + b * blk_len;
    int chosen[HX_WALK_CAND];
    int n = 0;
    if (b >= 1 && start <= N) {
        const int need = min(L, start - 1);
        for (int j = it - 1; j >= 0 && n < HX_WALK_CAND - 1; --j) {
            const uint8_t *pj = paths0 + (size_t)j * ((size_t)N + 1);
            bool fresh = true;
            for (int q = 0; q < n && fresh; ++q) {
                const uint8_t *pq = paths0 + (size_t)chosen[q] * ((size_t)N + 1);
                bool same = true;
                for (int i = lane; i < need; i += 32) same &= pj[start - 1 - i] == pq[start - 1 - i];
                if (__all_sync(0xffffffffu, same)) fresh = false;
            }
            if (fresh) chosen[n++] = j;
        }
    }
    if (lane == 0)
        for (int c = 1; c < HX_WALK_CAND; ++c) cand_idx[b * HX_WALK_CAND + c] = c - 1 < n ? chosen[c - 1] : -1;
}

template <int NIT>
__global__ void __launch_bounds__(32)
k_walk_q(const int32_t *__restrict__ termsq, const int32_t *__restrict__ logmq, const double *__restrict__ terms,
         const double *__restrict__ logm, int N, int L, int C, int blk_len, int warm, const uint8_t *__restrict__ guess,
         const uint8_t *paths0, const int *__restrict__ cand_idx, uint8_t *spec, int spec_stride, int *__restrict__ spec_ok,
         uint8_t *path, hx_dev_flags *__restrict__ df) {
    extern __shared__ __align__(128) unsigned char smraw[];
    __shared__ __align__(8) unsigned long long bars[3];
    const int lane = threadIdx.x;
    if (df->hole) return;
    const bool force_exact = df->q_unsafe != 0;
    if (lane == 0) TableRing<int32_t>::init(bars);
    __syncwarp();
    uint32_t bar_uses = 0;
    if (blockIdx.x == 0) {                                  // block 0 of the region: the walk proper
        const int end = min(N, blk_len);
        if (lane == 0) path[0] = HX_SYM_GAP;
        __syncwarp();
        const int hole = walk_q_range<NIT>(termsq, logmq, terms, logm, L, C, 1, end, path, path + 1, force_exact, smraw,
                                           bars, bar_uses);
        if (hole && lane == 0) { df->hole_site = hole; df->hole = 1; }
        if (!hole && lane == 0 && end == N) df->hole_site = 0;
        return;
    }
    // speculative walks: CTA 1 + (b-1)*CAND + c = block b >= 1 from candidate history c
    const int b = 1 + ((int)blockIdx.x - 1) / HX_WALK_CAND, c = ((int)blockIdx.x - 1) % HX_WALK_CAND;
    const int start = 1 + b * blk_len;
    if (start > N) return;
    const int end = min(N, start + blk_len - 1);
    const int s0 = max(1, start - warm);
    uint8_t *out = spec + ((size_t)b * HX_WALK_CAND + c) * spec_stride;     // out[snp - s0]
    int hole;
    if (c == 0) {
        // from the majority alleles, `warm` sites early so that the walk's own choices fill the lookback window
        hole = walk_q_range<NIT>(termsq, logmq, terms, logm, L, C, s0, end, guess, out, force_exact, smraw, bars, bar_uses);
    } else {
        const int j = cand_idx[b * HX_WALK_CAND + c];
        if (j < 0) { if (lane == 0) spec_ok[b * HX_WALK_CAND + c] = 0; return; }
        // from an earlier haplotype's choices right before the block (the walk often retraces a strain it has found)
        const uint8_t *cand = paths0 + (size_t)j * ((size_t)N + 1);
        hole = walk_q_range<NIT>(termsq, logmq, terms, logm, L, C, start, end, cand, out + (start - s0), force_exact, smraw,
                                 bars, bar_uses);
    }
    if (lane == 0) spec_ok[b * HX_WALK_CAND + c] = hole ? 0 : 1;
}

// Accepts or redoes the speculative blocks, in order (one warp; see k_walk_q).
template <int NIT>
__global__ void __launch_bounds__(32)
k_walk_fix(const int32_t *__restrict__ termsq, const int32_t *__restrict__ logmq, const double *__restrict__ terms,
           const double *__restrict__ logm, int N, int L, int C, int blk_len, int warm, int n_blocks,
           const uint8_t *paths0, const int *__restrict__ cand_idx, const uint8_t *__restrict__ spec, int spec_stride,
           const int *__restrict__ spec_ok, uint8_t *path, hx_dev_flags *__restrict__ df) {
    extern __shared__ __align__(128) unsigned char smraw[];
    __shared__ __align__(8) unsigned long long bars[3];
    const int lane = threadIdx.x;
    if (df->hole) return;
    const bool force_exact = df->q_unsafe != 0;
    if (lane == 0) TableRing<int32_t>::init(bars);
    __syncwarp();
    uint32_t bar_uses = 0;
    int redone = 0;                                          // sites walked again
    for (int b = 1; b < n_blocks; ++b) {
        const int start = 1 + b * blk_len;
        if (start > N) break;
        const int end = min(N, start + blk_len - 1);
        const int s0 = max(1, start - warm);
        // A speculative walk of the block is the sequential walk's continuation iff the history it assumed agrees with
        // the final path on the L sites before the block (a site only sees L symbols back).
        const int need = min(L, start - 1);
        int hit = -1;
        for (int c = 0; c < HX_WALK_CAND && hit < 0; ++c) {
            if (!spec_ok[b * HX_WALK_CAND + c]) continue;
            const uint8_t *sp = spec + ((size_t)b * HX_WALK_CAND + c) * spec_stride;
            bool same = true;
            if (c == 0) {
                if (s0 > 1) {                               // (a walk that started at site 1 had the true history)
                    if (start - need < s0) continue;        // the warm-up must cover the whole lookback
                    for (int i = lane; i < need; i += 32) same &= sp[start - 1 - i - s0] == path[start - 1 - i];
                }
            } else {
                const uint8_t *cand = paths0 + (size_t)cand_idx[b * HX_WALK_CAND + c] * ((size_t)N + 1);
                for (int i = lane; i < need; i += 32) same &= cand[start - 1 - i] == path[start - 1 - i];
            }
            if (__all_sync(0xffffffffu, same)) hit = c;
        }
        if (hit >= 0) {
            const uint8_t *sp = spec + ((size_t)b * HX_WALK_CAND + hit) * spec_stride;
            for (int snp = start + lane; snp <= end; snp += 32) path[snp] = sp[snp - s0];
            __syncwarp();
            __threadfence_block();
            continue;
        }
        // No candidate started from the right history: walk the block from the final path - but only until it falls
        // in step with one of the speculative walks (agreement on L consecutive sites is agreement for good).
        const int SUB = L > 48 ? L : 48;
        for (int sub = start; sub <= end; sub += SUB) {
            const int e = min(end, sub + SUB - 1);
            __syncwarp();
            __threadfence();                                 // path[] written by this warp is read as history
            const int hole = walk_q_range<NIT>(termsq, logmq, terms, logm, L, C, sub, e, path, path + sub, force_exact,
                                               smraw, bars, bar_uses);
            if (hole) {
                if (lane == 0) { df->hole_site = hole; df->hole = 1; }
                return;
            }
            redone += e - sub + 1;
            __syncwarp();
            __threadfence_block();
            if (e == end || e - L + 1 < start) continue;
            int join = -1;
            for (int c = 0; c < HX_WALK_CAND && join < 0; ++c) {
                if (!spec_ok[b * HX_WALK_CAND + c]) continue;
                const uint8_t *sp = spec + ((size_t)b * HX_WALK_CAND + c) * spec_stride;
                bool same = true;
                for (int i = lane; i < L; i += 32) same &= path[e - i] == sp[e - i - s0];
                if (__all_sync(0xffffffffu, same)) join = c;
            }
            if (join >= 0) {
                const uint8_t *sp = spec + ((size_t)b * HX_WALK_CAND + join) * spec_stride;
                for (int snp = e + 1 + lane; snp <= end; snp += 32) path[snp] = sp[snp - s0];
                __syncwarp();
                __threadfence_block();
                break;
            }
        }
    }
    if (lane == 0) { df->hole_site = 0; df->walk_redone += redone; }
}

// Wide-lookback walk (L*448 B per site does not fit the staged pipeline, e.g. ONT L ~ 300):
// one warp per candidate symbol, lanes split the lookbacks and combine with warp shuffles;
// warp 0 then takes the 7-way argmax (pick_site, as in k_walk_tables).
__global__ void __launch_bounds__(256)
k_walk_wide(const double *__restrict__ terms, const double *__restrict__ logm,
            const int32_t *__restrict__ vseen, int N, int L, int Lw, int flags,
            uint8_t *__restrict__ path, hx_dev_flags *__restrict__ df) {
    __shared__ uint8_t ring[HX_RING];
    __shared__ double s_lw[8];
    __shared__ int s_next;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;   // warp = candidate symbol (7 = idle helper)
    if (df->hole) return;
    if (threadIdx.x == 0) { ring[0] = HX_SYM_GAP; path[0] = HX_SYM_GAP; }
    __syncthreads();
    for (int snp = 1; snp <= N; ++snp) {
        const double *lmrow = logm + (int64_t)snp * 8;
        const unsigned cmask = (unsigned)lmrow[7];
        const int lmax = L < snp ? L : snp;
        const int lt = lmax < Lw ? lmax : Lw;
        const bool cand = warp < HX_NSYM && ((cmask >> warp) & 1u);
        if (cand) {
            const double *base = terms + ((int64_t)snp * Lw) * 56 + warp;
            double p = 0.0;
            for (int l = 1 + lane; l <= lt; l += 32)
                p += base[((l - 1) * HX_NSYM + ring[(snp - l) & (HX_RING - 1)]) * 8];
            p = add_beyond_band(p, vseen, flags, snp, lt + 1 + lane, lmax, 32);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) p += __shfl_xor_sync(0xffffffffu, p, o);
            if (lane == 0) s_lw[warp] = lmrow[warp] + p;
        } else if (lane == 0 && warp < 8) {
            s_lw[warp] = -INFINITY;
        }
        __syncthreads();
        if (warp == 0) {
            const int next = pick_site<true>(s_lw[lane & 7], cmask, lmrow, terms + ((int64_t)snp * Lw) * 56, ring, snp, lt,
                                             lmax, vseen, flags);
            if (lane == 0) {
                s_next = next;
                if (next >= 0) { ring[snp & (HX_RING - 1)] = (uint8_t)next; path[snp] = (uint8_t)next; }
            }
        }
        __syncthreads();
        if (s_next < 0) {                                  // gretel.py:176-180
            if (threadIdx.x == 0) { df->hole_site = snp; df->hole = 1; }
            return;
        }
    }
    if (threadIdx.x == 0) df->hole_site = 0;
}

// ---- per-site marginals of the chosen path, then ordered sums -------------------------
__global__ void k_path_stats(const double *__restrict__ scnt_cur, const double *__restrict__ scnt_orig,
                             int N, const uint8_t *__restrict__ path, double *__restrict__ site,
                             const hx_dev_flags *__restrict__ df) {
    const int snp = blockIdx.x * blockDim.x + threadIdx.x + 1;
    if (df->hole || snp > N) return;
    const int s = path[snp];
    const double m = scnt_cur[(int64_t)snp * 8 + s] / scnt_cur[(int64_t)snp * 8 + 7];
    const double to = scnt_orig[(int64_t)snp * 8 + 7];
    const double mo = to == 0 ? 0.0 : scnt_orig[(int64_t)snp * 8 + s] / to;
    const int64_t stride = (int64_t)N + 2;
    site[snp] = hx_gl_log10(m);
    site[stride + snp] = hx_gl_log10(mo);
    site[2 * stride + snp] = m;
}

// The minimum marginal is what the reweighting needs (ratio = max(min, min_remove), cmd.py:157-160): a parallel
// reduction on the main stream.  The two log10 sums are only reported; they are strictly ordered chains (same order
// as gretel.py:185-186) and run on a side stream while the reweighting and the next haplotype's tables proceed.
__global__ void __launch_bounds__(1024)
k_path_min(const double *__restrict__ site, int N, double min_remove, hx_hap_stats *__restrict__ stats,
           const hx_dev_flags *__restrict__ df) {
    __shared__ double sh[32];
    if (df->hole) { if (threadIdx.x == 0) stats->done = 0.0; return; }
    const double *m = site + 2 * ((int64_t)N + 2);
    double acc = INFINITY;
    for (int x = 1 + threadIdx.x; x <= N; x += 1024) { const double v = m[x]; acc = v < acc ? v : acc; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const double v = __shfl_xor_sync(0xffffffffu, acc, o); acc = v < acc ? v : acc; }
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; ++w) acc = sh[w] < acc ? sh[w] : acc;
        stats->min_marginal = acc;
        stats->ratio = acc < min_remove ? min_remove : acc;    // cmd.py:157-160
        stats->done = 1.0;
    }
}

// Two threads each run one strictly ordered accumulation out of shared memory while warps 2..7 stage the next
// block of per-site values, so the ordered adds never wait on HBM.
constexpr int HX_SUM_CH = 896;

__global__ void __launch_bounds__(256)
k_path_sum(const double *__restrict__ site, int N, hx_hap_stats *__restrict__ stats) {
    __shared__ double buf[2][2][HX_SUM_CH];
    const int tid = threadIdx.x;
    if (stats->done != 1.0) return;                            // the walk found a hole (k_path_min): nothing to sum
    const int64_t stride = (int64_t)N + 2;
    const int nch = (N + HX_SUM_CH - 1) / HX_SUM_CH;
    auto stage = [&](int c, int t0, int nt) {
        const int base = 1 + c * HX_SUM_CH;
        const int n = min(HX_SUM_CH, N - base + 1);
        for (int a = 0; a < 2; ++a)
            for (int x = t0; x < n; x += nt) buf[c & 1][a][x] = site[a * stride + base + x];
    };
    stage(0, tid, 256);
    __syncthreads();
    const int role = tid < 2 ? tid : -1;                       // two ordered sums in warp 0
    double acc = 0.0;
    for (int c = 0; c < nch; ++c) {
        if (tid >= 64) {
            if (c + 1 < nch) stage(c + 1, tid - 64, 192);
        } else if (role >= 0) {
            const int n = min(HX_SUM_CH, N - c * HX_SUM_CH);
            const double *p = buf[c & 1][role];
            int x = 0;
            for (; x + 8 <= n; x += 8) {                       // loads first, then the ordered chain
                double v[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) v[q] = p[x + q];
#pragma unroll
                for (int q = 0; q < 8; ++q) acc += v[q];
            }
            for (; x < n; ++x) acc += p[x];
        }
        __syncthreads();
    }
    if (role == 0) stats->hp_current = acc;
    if (role == 1) stats->hp_original = acc;
}

// ---- reweight ---------------------------------------------------------------------------
// One thread per band cell (pj,d) on the path.  Closed form of the loop nest in
// gretel.py:79-98: pairs (p,q) with q<=N-1 once, adjacent pairs (i,i+1), i<=N-2, twice
// (two sequential roundings), (N-1,N) once, (p,N) with p<=N-2 never, (N,N+1) once with
// symbols (path[N], '_').
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK)
k_reweight_path(float *__restrict__ band, int N, int W, const uint8_t *__restrict__ path,
                const double *__restrict__ ratio_ptr, double ratio_val,
                double *__restrict__ partials, const hx_dev_flags *__restrict__ df) {
    __shared__ double sh[BLOCK / 32];
    double removed = 0.0;
    const bool dead = df->hole != 0;
    const int64_t idx = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    const int64_t pj = 1 + idx / W;
    const int d = 1 + (int)(idx % W);
    const int64_t pi = pj - d;
    if (!dead && pj <= (int64_t)N + 1 && pi >= 0) {
        int times;
        if (pj <= N - 1) times = d == 1 ? 2 : 1;
        else times = d == 1 ? 1 : 0;
        if (times) {
            const double ratio = ratio_ptr ? *ratio_ptr : ratio_val;
            const unsigned a = path[pi];
            const unsigned b = pj == (int64_t)N + 1 ? (unsigned)HX_SYM_GAP : (unsigned)path[pj];
            float *p = band + hx_cell_off(W, pi, pj) + a * HX_NSYM + b;
            double old = (double)*p;
            for (int t = 0; t < times; ++t) {
                const double nw = old - (ratio * old);
                const float stored = (float)nw;
                removed += old - nw;
                old = (double)stored;
            }
            *p = (float)old;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) removed += __shfl_xor_sync(0xffffffffu, removed, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = removed;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < BLOCK / 32; ++w) t += sh[w];
        partials[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(1024)
k_sum_partials(const double *__restrict__ partials, int64_t n, double *__restrict__ out) {
    __shared__ double sh[32];
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) acc += partials[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 32; ++w) t += sh[w];
        *out = t;
    }
}

__global__ void k_reweight_matrix(float *__restrict__ band, int64_t n, double ratio) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const double old = (double)band[i];
        band[i] = (float)(old - ratio * old);
    }
}

int launch_reweight(hx_matrix *h, const uint8_t *d_path, const double *d_ratio, double ratio,
                    double *d_removed) {
    constexpr int BLOCK = 256;
    const int64_t cells = ((int64_t)h->N + 1) * h->W;
    const int64_t grid = (cells + BLOCK - 1) / BLOCK;
    HX_CUDA(h->d_partials.grow(grid * (int64_t)sizeof(double), h->stream));
    k_reweight_path<BLOCK><<<(unsigned)grid, BLOCK, 0, h->stream>>>(h->band.p, h->N, h->W, d_path, d_ratio,
                                                                    ratio, h->d_partials.p, h->d_flags.p);
    k_sum_partials<<<1, 1024, 0, h->stream>>>(h->d_partials.p, grid, d_removed);
    h->use.launches += 2;
    h->use.counts_dirty = true;
    HX_CUDA(cudaGetLastError());
    return HX_OK;
}

// What the recovery entry points do before their walks: room for the paths and the stats of n haplotypes, orig's
// counts (produced on orig's stream) ordered before the walk, the walk flags and the stats cleared (`done` must start
// at 0 for the hole test of the ordered sums), the timing started.
int recovery_prologue(hx_matrix *cur, hx_matrix *orig, int64_t path_bytes, int n) {
    HX_CUDA(cur->d_path.grow(path_bytes, cur->stream));
    HX_CUDA(cur->d_stats.grow(n * (int64_t)sizeof(hx_hap_stats), cur->stream));
    if (orig->stream != cur->stream && orig->use.counts_dirty) {
        const int rc = hx_ensure_counts(orig);
        if (rc) return rc;
        HX_CUDA(cudaStreamSynchronize(orig->stream));
    }
    HX_CUDA(cudaMemsetAsync(cur->d_flags.p, 0, offsetof(hx_dev_flags, walk_redone), cur->stream));
    HX_CUDA(cudaMemsetAsync(cur->d_stats.p, 0, n * sizeof(hx_hap_stats), cur->stream));
    HX_CUDA(cudaEventRecord(cur->ev0, cur->stream));
    return HX_OK;
}

// ... and after them: the ordered sums of every haplotype joined into the main stream, the timing stopped, the stats of
// n haplotypes, path_bytes of paths and (if `hole` is given) the hole flags copied back.
int recovery_epilogue(hx_matrix *cur, hx_hap_stats *stats, int n, uint8_t *paths, int64_t path_bytes,
                      hx_dev_flags *hole) {
    for (int b = 0; b < 2; ++b)
        if (cur->use.sum_busy[b]) { HX_CUDA(cudaStreamWaitEvent(cur->stream, cur->sum_done[b], 0)); cur->use.sum_busy[b] = false; }
    HX_CUDA(cudaEventRecord(cur->ev1, cur->stream));
    cur->use.ev_rec = true;
    if (hole)
        HX_CUDA(cudaMemcpyAsync(hole, cur->d_flags.p, offsetof(hx_dev_flags, q_unsafe), cudaMemcpyDeviceToHost, cur->stream));
    HX_CUDA(cudaMemcpyAsync(stats, cur->d_stats.p, n * sizeof(hx_hap_stats), cudaMemcpyDeviceToHost, cur->stream));
    HX_CUDA(cudaMemcpyAsync(paths, cur->d_path.p, (size_t)path_bytes, cudaMemcpyDeviceToHost, cur->stream));
    HX_CUDA(cudaStreamSynchronize(cur->stream));
    cudaEventElapsedTime(&cur->use.last_ms[1], cur->ev0, cur->ev1);
    return HX_OK;
}

int launch_generate(hx_matrix *cur, hx_matrix *orig, int L, int flags, uint8_t *d_path,
                    hx_hap_stats *d_stats, double min_remove, int it = 0, int n_prev = 0) {
    int rc = hx_ensure_counts(cur);
    if (rc) return rc;
    rc = hx_ensure_counts(orig);
    if (rc) return rc;
    const int N = cur->N;
    const int64_t sites = (int64_t)N + 2;
    const int Lw = L < cur->W ? (L < 1 ? 1 : L) : cur->W;          // lookbacks that stay inside the band
    // float64 tables, then (quantised walk only) their int32 fixed-point twins with Lq >= L rows per site
    const bool use_q = L >= 1 && L <= 32 && L <= cur->W;
    const int nit = use_q ? (L - 1 + 3) / 4 : 0;
    const int Lq = use_q ? 4 * nit + 1 : 0;
    HX_CUDA(cur->terms.grow(sites * Lw * HX_NSYM * 8 * (int64_t)sizeof(double), cur->stream));
    HX_CUDA(cur->logm.grow(sites * 8 * (int64_t)sizeof(double), cur->stream));
    if (use_q) {
        HX_CUDA(cur->termsq.grow(sites * Lq * HX_NSYM * 8 * (int64_t)sizeof(int32_t), cur->stream));
        HX_CUDA(cur->logmq.grow(sites * 8 * (int64_t)sizeof(int32_t), cur->stream));
    }
    const double *terms = cur->terms.p, *logm = cur->logm.p;
    int32_t *termsq = use_q ? cur->termsq.p : nullptr;
    int32_t *logmq = use_q ? cur->logmq.p : nullptr;
    hx_dev_flags *df = cur->d_flags.p;
    const int64_t tthreads = (int64_t)(N + 1) * (Lw > Lq ? Lw : Lq) * 8;
    k_walk_terms<<<(unsigned)((tthreads + 255) / 256), 256, 0, cur->stream>>>(cur->band.p, cur->vseen.p, N, cur->W, Lw,
                                                                              flags, cur->terms.p, termsq, Lq,
                                                                              &df->q_unsafe);
    // parallel-in-time walk (k_walk_q): blocks of sites walked concurrently from a guessed history, then verified
    int n_blocks = 1, blk_len = N > 0 ? N : 1, warm = 0;
    static const int blocks_env = getenv("HX_WALK_BLOCKS") ? atoi(getenv("HX_WALK_BLOCKS")) : 0;   // 1 = sequential
    if (use_q && N >= 1024 && blocks_env != 1) {
        warm = 4 * L > 64 ? 4 * L : 64;
        const int want = blocks_env > 1 ? blocks_env : 24;      // 1 + 23 x HX_WALK_CAND CTAs of one warp: one wave on 148 SMs
        blk_len = (N + want - 1) / want;
        if (blk_len < 2 * warm) blk_len = 2 * warm;
        n_blocks = (N + blk_len - 1) / blk_len;
    }
    const int spec_stride = blk_len + warm;
    const int64_t n_starts = (int64_t)n_blocks * HX_WALK_CAND;
    HX_CUDA(cur->spec.grow(n_starts * spec_stride, cur->stream));
    HX_CUDA(cur->guess.grow(sites, cur->stream));
    HX_CUDA(cur->spec_ok.grow(n_starts * (int64_t)sizeof(int), cur->stream));
    HX_CUDA(cur->cand_idx.grow(n_starts * (int64_t)sizeof(int), cur->stream));
    uint8_t *spec = cur->spec.p, *guess = cur->guess.p;
    int *spec_ok = cur->spec_ok.p, *cand_idx = cur->cand_idx.p;
    const uint8_t *paths0 = d_path - (size_t)n_prev * ((size_t)N + 1);              // the haplotypes found so far (hx_recover)
    k_walk_logm<<<(N + 1 + 127) / 128, 128, 0, cur->stream>>>(cur->scnt.p, N, flags, cur->logm.p, logmq, guess);
    if (n_blocks > 1) {
        k_walk_pick<<<n_blocks, 32, 0, cur->stream>>>(paths0, n_prev, N, L, blk_len, cand_idx);
        cur->use.launches++;
    }
    // sites per staged chunk: three chunks (terms + log-marginals) must fit in shared memory
    const int64_t site_bytes = (int64_t)Lw * 448 + 64;
    int C = (int)((200 * 1024) / (3 * site_bytes));
    if (C > 64) C = 64;
    if (use_q) {
        const int64_t qsite = (int64_t)Lq * 224 + 32;
        int Cq = (int)((200 * 1024) / (3 * qsite));
        if (Cq > 128) Cq = 128;
        const size_t qsmem = (size_t)3 * Cq * qsite;
#define HX_WALK_Q(NIT)                                                                                              \
    case NIT:                                                                                                       \
        HX_CUDA(cudaFuncSetAttribute(k_walk_q<NIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qsmem));      \
        k_walk_q<NIT><<<1 + (n_blocks - 1) * HX_WALK_CAND, 32, qsmem, cur->stream>>>(                                  \
            termsq, logmq, terms, logm, N, L, Cq, blk_len, warm, guess, paths0, cand_idx, spec, spec_stride, spec_ok,   \
            d_path, df);                                                                                            \
        if (n_blocks > 1) {                                                                                         \
            HX_CUDA(cudaFuncSetAttribute(k_walk_fix<NIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qsmem)); \
            k_walk_fix<NIT><<<1, 32, qsmem, cur->stream>>>(termsq, logmq, terms, logm, N, L, Cq, blk_len, warm,        \
                                                           n_blocks, paths0, cand_idx, spec, spec_stride, spec_ok,     \
                                                           d_path, df);                                                 \
            cur->use.launches++;                                                                                    \
        }                                                                                                           \
        break;
        switch (nit) {
            HX_WALK_Q(0) HX_WALK_Q(1) HX_WALK_Q(2) HX_WALK_Q(3) HX_WALK_Q(4) HX_WALK_Q(5) HX_WALK_Q(6) HX_WALK_Q(7)
            HX_WALK_Q(8)
        }
#undef HX_WALK_Q
    } else if (C < 1) {
        k_walk_wide<<<1, 256, 0, cur->stream>>>(terms, logm, cur->vseen.p, N, L, Lw, flags, d_path, df);
    } else {
        const size_t wsmem = (size_t)3 * C * site_bytes;
        HX_CUDA(cudaFuncSetAttribute(k_walk_tables, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
        k_walk_tables<<<1, 32, wsmem, cur->stream>>>(terms, logm, cur->vseen.p, N, L, Lw, flags, C, d_path, df);
    }
    cur->use.launches += 2;
    // per-site values of this haplotype: two alternating buffers, so that the ordered sums of haplotype `it` (side
    // stream) may still be running while haplotype it+1 is walked
    double *site = cur->d_site.p + (size_t)(it & 1) * 3 * ((size_t)N + 2);
    if (!cur->sum_stream) {
        HX_CUDA(cudaStreamCreateWithFlags(&cur->sum_stream, cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) HX_CUDA(cudaEventCreateWithFlags(&cur->sum_done[b], cudaEventDisableTiming));
        HX_CUDA(cudaEventCreateWithFlags(&cur->site_ready, cudaEventDisableTiming));
    }
    if (cur->use.sum_busy[it & 1]) HX_CUDA(cudaStreamWaitEvent(cur->stream, cur->sum_done[it & 1], 0));
    k_path_stats<<<(N + 255) / 256, 256, 0, cur->stream>>>(cur->scnt.p, orig->scnt.p, N, d_path, site, df);
    k_path_min<<<1, 1024, 0, cur->stream>>>(site, N, min_remove, d_stats, df);
    HX_CUDA(cudaEventRecord(cur->site_ready, cur->stream));
    HX_CUDA(cudaStreamWaitEvent(cur->sum_stream, cur->site_ready, 0));
    k_path_sum<<<1, 256, 0, cur->sum_stream>>>(site, N, d_stats);
    HX_CUDA(cudaEventRecord(cur->sum_done[it & 1], cur->sum_stream));
    cur->use.sum_busy[it & 1] = true;
    cur->use.launches += 4;
    HX_CUDA(cudaGetLastError());
    return HX_OK;
}

}  // namespace

// how many speculative walk blocks had to be walked again so far (diagnostics; tools/ and tests)
extern "C" int hx_debug_walk_redone(hx_matrix *h, int *n) {
    if (!h || !n) return HX_E_ARG;
    if (cudaSetDevice(h->device) != cudaSuccess) return HX_E_CUDA;
    if (cudaMemcpyAsync(n, &h->d_flags.p->walk_redone, sizeof(int), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) return HX_E_CUDA;
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) return HX_E_CUDA;
    return HX_OK;
}

int hx_ensure_counts(hx_matrix *h) {
    if (!h->use.counts_dirty) return HX_OK;
    k_site_counts<<<(h->N + 1 + 127) / 128, 128, 0, h->stream>>>(h->band.p, h->N, h->W, h->scnt.p, h->vseen.p);
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    h->use.counts_dirty = false;
    return HX_OK;
}

// --------------------------------------------------------------------------- C ABI
extern "C" {

int hx_counts_all(hx_matrix *h, double *out) {
    HX_CHECK_ARG(h && out);
    HX_CUDA(cudaSetDevice(h->device));
    int rc = hx_ensure_counts(h);
    if (rc) return rc;
    HX_CUDA(cudaMemcpyAsync(out, h->scnt.p, sizeof(double) * 8 * ((size_t)h->N + 1), cudaMemcpyDeviceToHost,
                            h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    return HX_OK;
}

int hx_marginal_of_at(hx_matrix *h, int sym, int32_t pos, double *out) {
    HX_CHECK_ARG(h && out && sym >= 0 && sym < HX_NSYM && pos >= 0 && pos <= h->N);
    HX_CUDA(cudaSetDevice(h->device));
    int rc = hx_ensure_counts(h);
    if (rc) return rc;
    double row[8];
    HX_CUDA(cudaMemcpyAsync(row, h->scnt.p + (size_t)pos * 8, sizeof(row), cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    *out = row[7] == 0 ? 0.0 : row[sym] / row[7];
    return HX_OK;
}

int hx_edge_weights_at(hx_matrix *h, int32_t snp, const uint8_t *path, int32_t L, int flags,
                       double weights[7], double *total, int *mask) {
    HX_CHECK_ARG(h && path && weights && total && mask && snp >= 1 && snp <= h->N && L >= 0);
    HX_CUDA(cudaSetDevice(h->device));
    int rc = hx_ensure_counts(h);
    if (rc) return rc;
    HX_CUDA(h->d_path.grow((int64_t)h->N + 2, h->stream));
    HX_CUDA(cudaMemcpyAsync(h->d_path.p, path, (size_t)snp, cudaMemcpyHostToDevice, h->stream));
    k_edge_one<<<1, 32, 0, h->stream>>>(h->band.p, h->scnt.p, h->vseen.p, h->W, L, flags, snp, h->d_path.p, h->d_misc.p);
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    double res[9];
    HX_CUDA(cudaMemcpyAsync(res, h->d_misc.p, sizeof(res), cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    for (int s = 0; s < 7; ++s) weights[s] = res[s];
    *total = res[7];
    *mask = (int)res[8];
    return HX_OK;
}

int hx_generate_path(hx_matrix *cur, hx_matrix *orig, int32_t L, int flags, uint8_t *out_path,
                     double out[3], int32_t *hole_site) {
    HX_CHECK_ARG(cur && orig && out_path && out && hole_site);
    HX_CHECK_ARG(cur->N == orig->N && cur->device == orig->device && L >= 0 && L <= HX_MAX_L);
    HX_CUDA(cudaSetDevice(cur->device));
    const int64_t N = cur->N;
    int rc = recovery_prologue(cur, orig, N + 2, 1);
    if (rc) return rc;
    rc = launch_generate(cur, orig, L, flags, cur->d_path.p, cur->d_stats.p, 0.0);
    if (rc) return rc;
    hx_hap_stats st;
    hx_dev_flags hf;
    rc = recovery_epilogue(cur, &st, 1, out_path, N + 1, &hf);
    if (rc) return rc;
    if (hf.hole) {
        *hole_site = hf.hole_site;
        return HX_HOLE;
    }
    *hole_site = 0;
    out[0] = st.hp_current; out[1] = st.hp_original; out[2] = st.min_marginal;
    return HX_OK;
}

int hx_reweight_path(hx_matrix *h, const uint8_t *path, double ratio, double *removed) {
    HX_CHECK_ARG(h && path && removed);
    HX_CUDA(cudaSetDevice(h->device));
    HX_CUDA(h->d_path.grow((int64_t)h->N + 2, h->stream));
    HX_CUDA(cudaMemsetAsync(h->d_flags.p, 0, offsetof(hx_dev_flags, walk_redone), h->stream));
    HX_CUDA(cudaMemcpyAsync(h->d_path.p, path, (size_t)h->N + 1, cudaMemcpyHostToDevice, h->stream));
    HX_CUDA(cudaEventRecord(h->ev0, h->stream));
    const int rc = launch_reweight(h, h->d_path.p, nullptr, ratio, h->d_misc.p);
    if (rc) return rc;
    HX_CUDA(cudaEventRecord(h->ev1, h->stream));
    h->use.ev_rec = true;
    HX_CUDA(cudaMemcpyAsync(removed, h->d_misc.p, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    HX_CUDA(cudaStreamSynchronize(h->stream));
    cudaEventElapsedTime(&h->use.last_ms[2], h->ev0, h->ev1);
    return HX_OK;
}

int hx_recover(hx_matrix *cur, hx_matrix *orig, int32_t L, int flags, int32_t max_paths,
               double min_remove, uint8_t *paths, double *stats, int32_t *n_found) {
    HX_CHECK_ARG(cur && orig && paths && stats && n_found && max_paths >= 0);
    HX_CHECK_ARG(cur->N == orig->N && cur->device == orig->device && L >= 0 && L <= HX_MAX_L);
    HX_CUDA(cudaSetDevice(cur->device));
    const int64_t N = cur->N;
    *n_found = 0;
    if (max_paths == 0) return HX_OK;
    int rc = recovery_prologue(cur, orig, (N + 1) * max_paths, max_paths);
    if (rc) return rc;
    for (int it = 0; it < max_paths; ++it) {
        uint8_t *dp = cur->d_path.p + (size_t)it * (N + 1);
        hx_hap_stats *ds = cur->d_stats.p + it;
        rc = launch_generate(cur, orig, L, flags, dp, ds, min_remove, it, it);
        if (rc) return rc;
        rc = launch_reweight(cur, dp, &ds->ratio, 0.0, &ds->removed);
        if (rc) return rc;
    }
    hx_hap_stats *hs = (hx_hap_stats *)malloc(sizeof(hx_hap_stats) * (size_t)max_paths);
    if (!hs) return HX_E_NOMEM;
    rc = recovery_epilogue(cur, hs, max_paths, paths, (N + 1) * max_paths, nullptr);
    int found = 0;
    for (; !rc && found < max_paths && hs[found].done == 1.0; ++found) {
        const hx_hap_stats &h = hs[found];
        double *o = stats + (size_t)found * 5;          // hanselx.h: hp_current, hp_original, min_marginal, ratio, removed
        o[0] = h.hp_current; o[1] = h.hp_original; o[2] = h.min_marginal; o[3] = h.ratio; o[4] = h.removed;
    }
    free(hs);
    if (rc) return rc;
    *n_found = found;
    return HX_OK;
}

int hx_reweight_matrix(hx_matrix *h, double ratio) {
    HX_CHECK_ARG(h);
    HX_CUDA(cudaSetDevice(h->device));
    const int64_t n = h->band_elems;
    k_reweight_matrix<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->band.p, n, ratio);
    h->use.launches++;
    h->use.counts_dirty = true;
    HX_CUDA(cudaGetLastError());
    return HX_OK;
}

}  // extern "C"

// ---- diagnostic: the device's log10 / 10**x on host arrays (hanselx.h) ---------------------------------------------
namespace {
__global__ void k_device_math(const double *__restrict__ x, double *__restrict__ y, int64_t n, int which) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = which ? hx_gl_pow10(x[i]) : hx_gl_log10(x[i]);
}
}  // namespace

extern "C" int hx_device_math(int32_t device, int which, const double *x, double *y, int64_t n) {
    HX_CHECK_ARG(x && y && n >= 0 && (which == 0 || which == 1));
    if (n == 0) return HX_OK;
    HX_CUDA(cudaSetDevice(device));
    double *dx = nullptr, *dy = nullptr;
    HX_CUDA(cudaMalloc((void **)&dx, sizeof(double) * (size_t)n));
    if (cudaMalloc((void **)&dy, sizeof(double) * (size_t)n) != cudaSuccess) { cudaFree(dx); hx_set_error("hx_device_math: out of memory"); return HX_E_NOMEM; }
    cudaError_t e = cudaMemcpy(dx, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        k_device_math<<<(unsigned)((n + 255) / 256), 256>>>(dx, dy, n, which);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(y, dy, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost);
    cudaFree(dx);
    cudaFree(dy);
    if (e != cudaSuccess) { hx_set_error("hx_device_math: %s", cudaGetErrorString(e)); return HX_E_CUDA; }
    return HX_OK;
}
