// The branch-weight arithmetic of Hansel.get_edge_weights_at shared by the recovery walk (recover.cu) and path
// scoring (score.cu): the lookback terms, the terms beyond the band, one candidate lane's weight, the ordered
// normalisation and first-max pick, and the path-independent walk tables.  Float64 on float32-stored cells in the
// operation order of oracle/hansel_oracle.c; both files are compiled with -fmad=false and evaluate log10 and 10**x
// exactly as glibc does (glibc_math.cuh), so that every caller gets the same bits.
#pragma once
#include <limits.h>
#include <math.h>

#include "hx_internal.cuh"
#include "glibc_math.cuh"

namespace {

// ---- the lookback terms of Hansel.get_edge_weights_at ------------------------------------
// log10((1 + H[a,s]) / (V + sum_a' H[a',s])) of one band cell, V valid symbols seen; 0.0 where the Laplace
// denominator is 0, i.e. the term is dropped.
__device__ __forceinline__ double lookback_term(const float *__restrict__ cell, unsigned a, int s, int v) {
    double sup = 0.0;
#pragma unroll
    for (int a2 = 0; a2 < HX_NSYM; ++a2) sup += (double)cell[a2 * HX_NSYM + s];
    const double den = (double)v + sup;
    return den != 0 ? hx_gl_log10((1.0 + (double)cell[a * HX_NSYM + s]) / den) : 0.0;
}

// acc + the terms of lookbacks l = from, from + step, ... <= lmax beyond the band, in that order.  Their cells are
// zero, so each term is log10(1 / V), dropped where V = 0.
__device__ __forceinline__ double add_beyond_band(double acc, const int32_t *__restrict__ vseen, int flags, int snp,
                                                  int from, int lmax, int step = 1) {
    for (int l = from; l <= lmax; l += step) {
        const int v = (flags & HX_F_VSITE_TO) ? vseen[snp] : vseen[snp - l];
        if (v != 0) acc += hx_gl_log10(1.0 / (double)v);
    }
    return acc;
}

// ---- branch weights at one site (lane = candidate symbol) ---------------------------------
// G lanes per site: G = 32 is one site per warp (lanes 0..6 = symbols), G = 8 four sites per warp (lanes g*8 + 0..6
// of group g).  Every lane of the warp calls it.  Returns this lane's unnormalised weight; *cand_mask gets the
// candidate set of its group (bit s = symbol s).
template <int G = 32>
__device__ __forceinline__ double edge_weight_lane(const float *__restrict__ band,
                                                   const double *__restrict__ scnt,
                                                   const int32_t *__restrict__ vseen, int W, int L,
                                                   int flags, int snp, const uint8_t *hist, unsigned *cand_mask) {
    const int lane = threadIdx.x & 31;
    const int s = lane & (G - 1);
    double c = 0.0;
    if (s < HX_NSYM) c = scnt[(int64_t)snp * 8 + s];
    const double total = scnt[(int64_t)snp * 8 + 7];
    const bool skip_unsym = !(flags & HX_F_KEEP_UNSYMBOLS);
    const bool cand = s < HX_NSYM && c > 0 && !(skip_unsym && (s == HX_SYM_N || s == HX_SYM_GAP));
    double ws = 0.0;
    if (cand) {
        double lw = hx_gl_log10(c / total);
        const int lmax = L < snp ? L : snp;
        const int lt = lmax < W ? lmax : W;
        const int v_to = vseen[snp];
        for (int l = 1; l <= lt; ++l) {
            const int pf = snp - l;
            lw += lookback_term(band + hx_cell_off(W, pf, snp), hist[pf], s, (flags & HX_F_VSITE_TO) ? v_to : vseen[pf]);
        }
        ws = hx_gl_pow10(add_beyond_band(lw, vseen, flags, snp, lt + 1, lmax));
    }
    static_assert(G == 32 || G == 8, "one site per warp or per 8 lanes");
    const unsigned ballot = __ballot_sync(0xffffffffu, cand);
    *cand_mask = G == 32 ? ballot : (ballot >> (lane & ~(G - 1))) & 0xffu;
    return ws;
}

// Sum in symbol order, normalise, first-max argmax (gretel.py:166-174) over the G-lane group of the calling lane.
template <int G = 32>
__device__ __forceinline__ int normalise_and_pick(double ws, unsigned cmask, double *wn_out,
                                                  double *tw_out) {
    double tw = 0.0;
#pragma unroll
    for (int s = 0; s < HX_NSYM; ++s) {
        const double v = __shfl_sync(0xffffffffu, ws, s, G);
        if ((cmask >> s) & 1u) tw += v;
    }
    const double wn = tw > 0 ? ws / tw : ws;
    int next = -1;
    double nv = 0.0;
#pragma unroll
    for (int s = 0; s < HX_NSYM; ++s) {
        const double v = __shfl_sync(0xffffffffu, wn, s, G);
        if ((cmask >> s) & 1u) {
            if (next < 0) { nv = v; next = s; }
            else if (v > nv) { nv = v; next = s; }
        }
    }
    *wn_out = wn;
    *tw_out = tw;
    return next;
}

// ---- walk tables: everything that does not depend on the path, computed in parallel ----
// terms[((snp*Lw + (l-1))*7 + a)*8 + s] = log10((1 + H[a,s,snp-l,snp]) / (V + sum_a' H[a',s,snp-l,snp]))
// (0.0 where the Laplace denominator is 0, i.e. the term is dropped), for every symbol a
// the path could hold at snp-l.  logm[snp*8+s] = log10(count_s / total); logm[snp*8+7] holds
// the candidate mask as a double.
#define HX_QSCALE 1048576.0      // fixed-point scale of the quantised walk tables (2^20)
#define HX_QSUNK (INT_MIN / 2)    // log weight of a non-candidate: below any real sum, far from overflow

// The int32 twin (quantised walk; termsq = nullptr and Lq = 0 without it) has Lq >= Lw rows per site; rows beyond
// Lw are zero so that every lane of k_walk_q owns a real row.  qflag[0] is raised if a term is too large for the
// fixed-point sums.
__global__ void k_walk_terms(const float *__restrict__ band, const int32_t *__restrict__ vseen, int N, int W,
                             int Lw, int flags, double *__restrict__ terms, int32_t *__restrict__ termsq, int Lq,
                             int *__restrict__ qflag) {
    const int Lr = Lw > Lq ? Lw : Lq;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t total = (int64_t)(N + 1) * Lr * 8;
    if (idx >= total) return;
    const int s = (int)(idx & 7);
    const int l = (int)((idx >> 3) % Lr) + 1;
    const int snp = (int)((idx >> 3) / Lr);
    double *out = l <= Lw ? terms + (((int64_t)snp * Lw + (l - 1)) * HX_NSYM) * 8 + s : nullptr;   // [snp][l][a][8]
    int32_t *outq = l <= Lq ? termsq + (((int64_t)snp * Lq + (l - 1)) * HX_NSYM) * 8 + s : nullptr;
    const int pf = snp - l;
    if (s >= HX_NSYM || snp < 1 || pf < 0 || l > Lw) {
#pragma unroll
        for (int a = 0; a < HX_NSYM; ++a) {
            if (out) out[a * 8] = 0.0;
            if (outq) outq[a * 8] = 0;
        }
        return;
    }
    const float *cell = band + hx_cell_off(W, pf, snp);
    const int v = (flags & HX_F_VSITE_TO) ? vseen[snp] : vseen[pf];
    bool unsafe = false;
#pragma unroll
    for (int a = 0; a < HX_NSYM; ++a) {
        const double t = lookback_term(cell, a, s, v);
        out[a * 8] = t;
        if (outq) {
            unsafe |= !(fabs(t) < 15.0);
            outq[a * 8] = __double2int_rn(fmax(fmin(t, 15.0), -15.0) * HX_QSCALE);
        }
    }
    if (unsafe) *qflag = 1;
}

// logmq and guess may be nullptr (the float64 tables only).
__global__ void k_walk_logm(const double *__restrict__ scnt, int N, int flags, double *__restrict__ logm,
                            int32_t *__restrict__ logmq, uint8_t *__restrict__ guess) {
    const int snp = blockIdx.x * blockDim.x + threadIdx.x;
    if (snp > N) return;
    const double total = scnt[(int64_t)snp * 8 + 7];
    const bool skip_unsym = !(flags & HX_F_KEEP_UNSYMBOLS);
    unsigned mask = 0;
    double gbest = -1.0;
    int gsym = snp == 0 ? HX_SYM_GAP : 0;                   // the majority allele: where a speculative block starts from
    for (int s = 0; s < HX_NSYM; ++s) {
        const double c = scnt[(int64_t)snp * 8 + s];
        const bool cand = c > 0 && !(skip_unsym && (s == HX_SYM_N || s == HX_SYM_GAP));
        if (cand && snp > 0 && c > gbest) { gbest = c; gsym = s; }
        const double lm = cand ? hx_gl_log10(c / total) : 0.0;
        logm[(int64_t)snp * 8 + s] = lm;
        if (logmq) logmq[(int64_t)snp * 8 + s] = cand ? __double2int_rn(lm * HX_QSCALE) : HX_QSUNK;
        if (cand) mask |= 1u << s;
    }
    logm[(int64_t)snp * 8 + 7] = (double)mask;
    if (logmq) logmq[(int64_t)snp * 8 + 7] = HX_QSUNK;
    if (guess) guess[snp] = (uint8_t)gsym;
}

}  // namespace
