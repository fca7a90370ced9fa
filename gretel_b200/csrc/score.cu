// K6: per-site branch weights and path likelihoods of given haplotypes (hx_score_paths; no reference counterpart,
// DESIGN.md §4 K6).  For haplotype h and site s the weights are exactly Hansel.get_edge_weights_at(s, p[h][0..s-1])
// (gretel.py:155), and the first-max pick over them is what generate_path would choose there (gretel.py:159-174).
// A path is given, so its lookback history is known at every site: the N sequential steps of the walk become
// H x N independent (haplotype, site) items.
//
// k_score_sites: 8 lanes per item (lane = candidate symbol), four items per warp; the normalisation and the pick are
// width-8 shuffles in symbol order (normalise_and_pick<8>).  A lane's log weight is summed in the reference's order
// either from the path-independent walk tables (k_walk_terms / k_walk_logm, built once per call and shared by all
// haplotypes: one table load per term) or, where those would not pay (L > 32 or L > W, e.g. ONT), straight from the
// band (edge_weight_lane<8>).  Both give the same bits.  k_score_sum then adds log10(w_hap) over the sites of one
// haplotype per thread, strictly in site order.
#include <stdlib.h>

#include <algorithm>

#include "hx_internal.cuh"
#include "glibc_math.cuh"
#include "recover_common.cuh"

namespace {

constexpr int SC_THREADS = 256;
constexpr int64_t SC_SCRATCH_MB = 256;      // tables + per-site scratch of one chunk of haplotypes
constexpr int SC_SITE_DOUBLES = 3;          // w_hap, w_second, log10(w_hap) per item (+ 8 with weights)

// A code > 6 at any site or anything but '_' at site 0 raises df->score_err.
__global__ void k_score_check(const uint8_t *__restrict__ haps, int64_t n, int N, hx_dev_flags *__restrict__ df) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t c = haps[i];
    const bool bad = i % ((int64_t)N + 1) == 0 ? c != HX_SYM_GAP : c > 6;
    if (bad) atomicOr(&df->score_err, 1);
}

// Item i = hl * N + (s - 1): site s of haplotype hl of the chunk (haps = the chunk's first path, N + 1 codes each).
// Outputs per item: w_hap, w_second, log10(w_hap) (0 where w_hap = 0) in site[0..2][item], best[item], and with
// `weights` the 7 normalised weights and the total.
template <bool TABLES>
__global__ void __launch_bounds__(SC_THREADS)
k_score_sites(const float *__restrict__ band, const double *__restrict__ scnt, const int32_t *__restrict__ vseen,
              const double *__restrict__ terms, const double *__restrict__ logm, int N, int W, int L, int Lw,
              int flags, const uint8_t *__restrict__ haps, int64_t n_items, double *__restrict__ site,
              uint8_t *__restrict__ best, double *__restrict__ weights) {
    const int q = threadIdx.x & 7;
    const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31);
    if ((t0 >> 3) >= n_items) return;                       // the whole warp is past the last item
    const int64_t mine = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    const bool live = mine < n_items;
    const int64_t item = live ? mine : n_items - 1;         // idle groups repeat the last item (shuffles need them)
    const int64_t hl = item / N;
    const int snp = (int)(item - hl * N) + 1;
    const uint8_t *path = haps + hl * ((int64_t)N + 1);
    unsigned cmask;
    double ws = 0.0;
    if (TABLES) {
        cmask = (unsigned)logm[(int64_t)snp * 8 + 7];
        if (q < HX_NSYM && ((cmask >> q) & 1u)) {
            // ((log10 P(s) + t1) + t2) + ... as edge_weight_lane adds them; a term is one table load
            double lw = logm[(int64_t)snp * 8 + q];
            const int lmax = L < snp ? L : snp;
            const int lt = lmax < Lw ? lmax : Lw;
            const double *base = terms + (int64_t)snp * Lw * 56 + q;
            for (int l = 1; l <= lt; ++l) lw += base[((l - 1) * HX_NSYM + path[snp - l]) * 8];
            ws = hx_gl_pow10(add_beyond_band(lw, vseen, flags, snp, lt + 1, lmax));
        }
    } else {
        ws = edge_weight_lane<8>(band, scnt, vseen, W, L, flags, snp, path, &cmask);
    }
    double wn, tw;
    const int pick = normalise_and_pick<8>(ws, cmask, &wn, &tw);
    const double w = q < HX_NSYM && ((cmask >> q) & 1u) ? wn : 0.0;
    const unsigned a = path[snp];                           // <= 6 (k_score_check)
    const double wh = __shfl_sync(0xffffffffu, w, (int)a, 8);
    double other = q == (int)a ? 0.0 : w;                   // the best of the other candidates
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) other = fmax(other, __shfl_xor_sync(0xffffffffu, other, o, 8));
    if (!live) return;
    if (weights) weights[item * 8 + q] = q < HX_NSYM ? w : tw;
    if (q == 0) {
        site[item] = wh;
        site[n_items + item] = other;
        best[item] = pick < 0 ? 255 : (uint8_t)pick;
    } else if (q == 1) {
        site[2 * n_items + item] = wh > 0 ? hx_gl_log10(wh) : 0.0;
    }
}

// One thread per haplotype of the chunk: loglik = sum of log10(w_hap) over the sites with w_hap > 0, in site order
// (left to right, float64, as a Python loop over math.log10 adds them); the sites with w_hap = 0; the sites whose
// pick is not the haplotype's allele.
__global__ void k_score_sum(const double *__restrict__ site, const uint8_t *__restrict__ best,
                            const uint8_t *__restrict__ haps, int N, int nh, int64_t n_items,
                            double *__restrict__ loglik, int32_t *__restrict__ n_unsup, int32_t *__restrict__ n_dis) {
    const int hl = blockIdx.x * blockDim.x + threadIdx.x;
    if (hl >= nh) return;
    const double *wh = site + (int64_t)hl * N;
    const double *lg = site + 2 * n_items + (int64_t)hl * N;
    const uint8_t *b = best + (int64_t)hl * N;
    const uint8_t *p = haps + (int64_t)hl * ((int64_t)N + 1) + 1;
    double acc = 0.0;
    int unsup = 0, dis = 0;
    int x = 0;
    for (; x + 8 <= N; x += 8) {                            // loads first, then the ordered chain
        double w[8], g[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { w[k] = wh[x + k]; g[k] = lg[x + k]; dis += b[x + k] != p[x + k]; }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (w[k] > 0) acc += g[k];
            else ++unsup;
        }
    }
    for (; x < N; ++x) {
        if (wh[x] > 0) acc += lg[x];
        else ++unsup;
        dis += b[x] != p[x];
    }
    loglik[hl] = acc;
    n_unsup[hl] = unsup;
    n_dis[hl] = dis;
}

int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

}  // namespace

void hx_score_free(hx_matrix *h) {
    cudaStream_t st = h->stream;
    h->sc_haps.release(st); h->sc_best.release(st); h->sc_site.release(st); h->sc_ll.release(st); h->sc_cnt.release(st);
    for (int e = 0; e < 2; ++e) {
        if (h->sc_ev[e]) cudaEventDestroy(h->sc_ev[e]);
        h->sc_ev[e] = nullptr;
    }
}

extern "C" int hx_score_paths(hx_matrix *h, const uint8_t *haps, int32_t n_haps, int32_t L, int flags,
                              double *weights, double *w_hap, double *w_second, uint8_t *best,
                              double *loglik, int32_t *n_unsupported, int32_t *n_disagree) {
    HX_CHECK_ARG(h && haps && n_haps >= 0 && L >= 0 && L <= HX_MAX_L);
    HX_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int N = h->N, W = h->W, H = n_haps;
    h->use.last_ms[4] = 0.0f;
    if (H == 0 || N < 1) return HX_OK;
    for (int e = 0; e < 2; ++e)
        if (!h->sc_ev[e]) HX_CUDA(cudaEventCreate(&h->sc_ev[e]));
    float ms = 0.0f;
    auto lap = [&]() -> int {                               // kernels enqueued since sc_ev[0] was recorded
        HX_CUDA(cudaGetLastError());
        HX_CUDA(cudaEventRecord(h->sc_ev[1], st));
        HX_CUDA(cudaEventSynchronize(h->sc_ev[1]));
        HX_CUDA(cudaEventElapsedTime(&ms, h->sc_ev[0], h->sc_ev[1]));
        h->use.last_ms[4] += ms;
        return HX_OK;
    };

    // the haplotypes, checked before anything reads them as table indices
    const int64_t path_bytes = (int64_t)H * (N + 1);
    HX_CUDA(h->sc_haps.grow(path_bytes, st));
    HX_CUDA(cudaMemcpyAsync(h->sc_haps.p, haps, (size_t)path_bytes, cudaMemcpyHostToDevice, st));
    hx_dev_flags *df = h->d_flags.p;
    HX_CUDA(cudaMemsetAsync(&df->score_err, 0, sizeof(int), st));
    HX_CUDA(cudaEventRecord(h->sc_ev[0], st));
    int rc = hx_ensure_counts(h);
    if (rc) return rc;
    k_score_check<<<(unsigned)((path_bytes + 255) / 256), 256, 0, st>>>(h->sc_haps.p, path_bytes, N, df);
    h->use.launches++;
    // path-independent tables: by default where recovery would take the fixed-point walk (L <= 32 inside the band);
    // HX_SCORE_TABLES=0/1 forces either way (tests: both give the same bits)
    const int Lw = L < W ? (L < 1 ? 1 : L) : W;
    const int tables_env = env_int("HX_SCORE_TABLES", -1);
    const bool tables = tables_env >= 0 ? tables_env != 0 : (L <= 32 && L <= W);
    int64_t table_bytes = 0;
    if (tables) {
        const int64_t sites = (int64_t)N + 2;
        table_bytes = sites * Lw * HX_NSYM * 8 * (int64_t)sizeof(double) + sites * 8 * (int64_t)sizeof(double);
        HX_CUDA(h->terms.grow(sites * Lw * HX_NSYM * 8 * (int64_t)sizeof(double), st));
        HX_CUDA(h->logm.grow(sites * 8 * (int64_t)sizeof(double), st));
        const int64_t tthreads = (int64_t)(N + 1) * Lw * 8;
        k_walk_terms<<<(unsigned)((tthreads + 255) / 256), 256, 0, st>>>(h->band.p, h->vseen.p, N, W, Lw, flags,
                                                                         h->terms.p, nullptr, 0, nullptr);
        k_walk_logm<<<(N + 1 + 127) / 128, 128, 0, st>>>(h->scnt.p, N, flags, h->logm.p, nullptr, nullptr);
        h->use.launches += 2;
    }
    rc = lap();
    if (rc) return rc;
    hx_dev_flags hf;
    HX_CUDA(cudaMemcpyAsync(&hf, df, sizeof(hf), cudaMemcpyDeviceToHost, st));
    HX_CUDA(cudaStreamSynchronize(st));
    if (hf.score_err) {
        hx_set_error("hx_score_paths: a haplotype code > 6, or site 0 is not '_'");
        return HX_E_ARG;
    }

    // haplotypes in chunks: the tables plus one chunk's per-site scratch stay within HX_SCORE_SCRATCH_MB
    const int64_t item_bytes = (SC_SITE_DOUBLES + (weights ? 8 : 0)) * (int64_t)sizeof(double) + 1;
    const int64_t budget = (int64_t)env_int("HX_SCORE_SCRATCH_MB", (int)SC_SCRATCH_MB) << 20;
    const int chunk = (int)std::max<int64_t>(1, std::min<int64_t>(H, (budget - table_bytes) / (item_bytes * N)));
    const int64_t cap_items = (int64_t)chunk * N;
    HX_CUDA(h->sc_site.grow(cap_items * (SC_SITE_DOUBLES + (weights ? 8 : 0)) * (int64_t)sizeof(double), st));
    HX_CUDA(h->sc_best.grow(cap_items, st));
    HX_CUDA(h->sc_ll.grow(H * (int64_t)sizeof(double), st));
    HX_CUDA(h->sc_cnt.grow(2 * H * (int64_t)sizeof(int32_t), st));
    for (int h0 = 0; h0 < H; h0 += chunk) {
        const int nh = std::min(chunk, H - h0);
        const int64_t n_items = (int64_t)nh * N;
        const uint8_t *dh = h->sc_haps.p + (int64_t)h0 * (N + 1);
        double *site = h->sc_site.p;
        double *dw = weights ? site + SC_SITE_DOUBLES * n_items : nullptr;
        const unsigned grid = (unsigned)((n_items * 8 + SC_THREADS - 1) / SC_THREADS);
        HX_CUDA(cudaEventRecord(h->sc_ev[0], st));
        if (tables)
            k_score_sites<true><<<grid, SC_THREADS, 0, st>>>(h->band.p, h->scnt.p, h->vseen.p, h->terms.p, h->logm.p,
                                                             N, W, L, Lw, flags, dh, n_items, site, h->sc_best.p, dw);
        else
            k_score_sites<false><<<grid, SC_THREADS, 0, st>>>(h->band.p, h->scnt.p, h->vseen.p, nullptr, nullptr, N,
                                                              W, L, Lw, flags, dh, n_items, site, h->sc_best.p, dw);
        k_score_sum<<<(nh + 127) / 128, 128, 0, st>>>(site, h->sc_best.p, dh, N, nh, n_items, h->sc_ll.p + h0,
                                                      h->sc_cnt.p + h0, h->sc_cnt.p + H + h0);
        h->use.launches += 2;
        rc = lap();
        if (rc) return rc;
        const int64_t o = (int64_t)h0 * N;
        if (w_hap) HX_CUDA(cudaMemcpyAsync(w_hap + o, site, sizeof(double) * n_items, cudaMemcpyDeviceToHost, st));
        if (w_second)
            HX_CUDA(cudaMemcpyAsync(w_second + o, site + n_items, sizeof(double) * n_items, cudaMemcpyDeviceToHost, st));
        if (best) HX_CUDA(cudaMemcpyAsync(best + o, h->sc_best.p, (size_t)n_items, cudaMemcpyDeviceToHost, st));
        if (weights)
            HX_CUDA(cudaMemcpyAsync(weights + o * 8, dw, sizeof(double) * 8 * n_items, cudaMemcpyDeviceToHost, st));
    }
    if (loglik) HX_CUDA(cudaMemcpyAsync(loglik, h->sc_ll.p, sizeof(double) * H, cudaMemcpyDeviceToHost, st));
    if (n_unsupported)
        HX_CUDA(cudaMemcpyAsync(n_unsupported, h->sc_cnt.p, sizeof(int32_t) * H, cudaMemcpyDeviceToHost, st));
    if (n_disagree)
        HX_CUDA(cudaMemcpyAsync(n_disagree, h->sc_cnt.p + H, sizeof(int32_t) * H, cudaMemcpyDeviceToHost, st));
    HX_CUDA(cudaStreamSynchronize(st));
    return HX_OK;
}
