// Bootstrap of the abundance EM (hx_em_bootstrap, DESIGN.md §4 K8): replicate 0 is K7's EM on the classes' counts,
// replicate b >= 1 the same EM on a multinomial resample of the T assigned reads over the classes, drawn by
// Philox4x32-10 keyed by the seed.  Both steps are exact: the resampled counts are integers that depend only on
// (count, seed, b), and the EM adds in the order hx_em_abundance fixes, so every replicate equals the host EM on the
// classes it keeps, bit for bit.
//
// k_boot_draw: one CTA per (replicate, slice of draw pairs); the class of a draw by binary search over the prefix sums
// of the counts, counted in a shared-memory histogram (global atomics when the classes do not fit), equal classes of a
// warp aggregated first.  k_boot_em: one CTA per replicate, persistent over its iterations: z per class, then one warp
// per haplotype computes its terms 32 at a time and adds them in class order, then the block-wide largest change.
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "glibc_math.cuh"
#include "hx_internal.cuh"

namespace {

constexpr int DRAW_THREADS = 256;
constexpr int DRAW_PAIRS_PER_THREAD = 64;            // a CTA draws up to 2 * 256 * 64 reads: its u32 histogram holds
constexpr uint64_t DRAW_PAIRS_PER_CTA = (uint64_t)DRAW_THREADS * DRAW_PAIRS_PER_THREAD;
constexpr int64_t DRAW_SMEM_CLASSES = 8192;          // classes whose prefix sums and histogram live in shared memory
constexpr int EM_THREADS = 1024;
constexpr int64_t EM_SMEM_BYTES = 200 * 1024;        // pi[H] and z[C] in shared memory up to this size
constexpr unsigned FULL = 0xffffffffu;

// Random123's philox4x32 with 10 rounds
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    }
    return c;
}

// the class c with P[c] <= u < P[c+1] (P[0] = 0 <= u < P[C] = T, P strictly ascending)
__device__ __forceinline__ int64_t class_of(const int64_t *P, int64_t C, uint64_t u) {
    int64_t lo = 0, hi = C;
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if ((uint64_t)P[mid] <= u) lo = mid;
        else hi = mid;
    }
    return lo;
}

// one draw per lane (c < 0: none); lanes that drew the same class add once.  The whole warp calls it.
template <bool SMEM>
__device__ __forceinline__ void count_draw(int64_t c, unsigned *s_hist, unsigned long long *row) {
    const unsigned peers = __match_any_sync(FULL, (unsigned long long)c);
    if (c < 0 || (int)(threadIdx.x & 31) != __ffs(peers) - 1) return;
    if (SMEM) atomicAdd(&s_hist[c], (unsigned)__popc(peers));
    else atomicAdd(&row[c], (unsigned long long)__popc(peers));
}

// Draw pairs [blockIdx.x * DRAW_PAIRS_PER_CTA, ...) of replicate b = rep0 + blockIdx.y into its row of cnt.
template <bool SMEM>
__global__ void __launch_bounds__(DRAW_THREADS)
k_boot_draw(const int64_t *__restrict__ pre, int64_t C, uint64_t T, uint64_t seed, int rep0,
            unsigned long long *__restrict__ cnt) {
    extern __shared__ unsigned long long s_draw[];
    int64_t *s_pre = reinterpret_cast<int64_t *>(s_draw);              // [C+1]
    unsigned *s_hist = reinterpret_cast<unsigned *>(s_pre + C + 1);    // [C]
    const int64_t *P = pre;
    if (SMEM) {
        for (int64_t c = threadIdx.x; c <= C; c += blockDim.x) s_pre[c] = pre[c];
        for (int64_t c = threadIdx.x; c < C; c += blockDim.x) s_hist[c] = 0;
        __syncthreads();
        P = s_pre;
    }
    const uint32_t b = (uint32_t)(rep0 + blockIdx.y);
    unsigned long long *row = cnt + (int64_t)blockIdx.y * C;
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    const uint64_t n_pairs = (T + 1) / 2, lo = (uint64_t)blockIdx.x * DRAW_PAIRS_PER_CTA;
    const uint64_t hi = min(n_pairs, lo + DRAW_PAIRS_PER_CTA);
    for (int k = 0; k < DRAW_PAIRS_PER_THREAD; ++k) {
        const uint64_t i0 = lo + (uint64_t)k * DRAW_THREADS;
        if (i0 >= hi) break;                                           // the same for the whole block
        const uint64_t i = i0 + threadIdx.x;
        int64_t ca = -1, cb = -1;
        if (i < hi) {
            const uint4 x = philox4x32_10(make_uint4((uint32_t)i, (uint32_t)(i >> 32), b, 0u), key);
            ca = class_of(P, C, __umul64hi(x.x | (uint64_t)x.y << 32, T));
            if (2 * i + 1 < T) cb = class_of(P, C, __umul64hi(x.z | (uint64_t)x.w << 32, T));
        }
        count_draw<SMEM>(ca, s_hist, row);
        count_draw<SMEM>(cb, s_hist, row);
    }
    if (SMEM) {
        __syncthreads();
        for (int64_t c = threadIdx.x; c < C; c += blockDim.x)
            if (s_hist[c]) atomicAdd(&row[c], (unsigned long long)s_hist[c]);
    }
}

// acc + the values v of the lanes with `take`, added one at a time in lane order.  The whole warp calls it.  The
// shuffles do not depend on acc, so unrolled they run ahead of the chain of additions.
__device__ __forceinline__ double add_in_lane_order(double acc, double v, bool take) {
    const unsigned m = __ballot_sync(FULL, take);
#pragma unroll
    for (int k = 0; k < 32; ++k) {
        const double x = __shfl_sync(FULL, v, k);
        if (m >> k & 1u) acc += x;
    }
    return acc;
}

// K7's EM on the classes with a count >= 1 of replicate r0 + blockIdx.x (row blockIdx.x of cnt), in
// hx_em_abundance's operation order: z_c in member order; acc[h] = the terms count_c * (pi[h] / z_c) added in class
// order (hoff/hcls list each haplotype's member entries in class order); pi[h] = acc[h] / T.  pi and z sit in shared
// memory if in_smem, else in the replicate's rows of g_pi / g_z.
__global__ void __launch_bounds__(EM_THREADS, 1)
k_boot_em(int H, int64_t C, const int64_t *__restrict__ class_off, const int32_t *__restrict__ members,
          const int64_t *__restrict__ hoff, const int32_t *__restrict__ hcls,
          const unsigned long long *__restrict__ cnt, double Td, int max_iter, double tol, bool in_smem,
          double *__restrict__ g_pi, double *__restrict__ g_z, int32_t *__restrict__ it_out,
          double *__restrict__ ll_out) {
    extern __shared__ double s_em[];
    __shared__ double s_max[EM_THREADS / 32];
    __shared__ double s_delta;
    const int r = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const unsigned long long *cb = cnt + (int64_t)r * C;
    double *pi = in_smem ? s_em : g_pi + (int64_t)r * H;
    double *z = in_smem ? s_em + H : g_z + (int64_t)r * C;
    const double p0 = 1.0 / H;
    for (int h = threadIdx.x; h < H; h += blockDim.x) pi[h] = p0;
    __syncthreads();
    double delta = INFINITY;
    int it = 0;
    while (it < max_iter) {
        ++it;
        for (int64_t c = threadIdx.x; c < C; c += blockDim.x) {
            if (!cb[c]) continue;
            double s = 0.0;
            for (int64_t j = class_off[c]; j < class_off[c + 1]; ++j) s += pi[members[j]];
            z[c] = s;
        }
        __syncthreads();
        double wmax = 0.0;
        for (int h = warp; h < H; h += nwarps) {
            const double ph = pi[h];
            double acc = 0.0;
            const int64_t e1 = hoff[h + 1];
            // the class and count of the next chunk's entry are loaded while this chunk's terms are added
            int32_t c_nx = 0;
            unsigned long long n_nx = 0;
            if (hoff[h] + lane < e1) { c_nx = hcls[hoff[h] + lane]; n_nx = cb[c_nx]; }
            for (int64_t e0 = hoff[h]; e0 < e1; e0 += 32) {
                const int32_t c = c_nx;
                const unsigned long long n = n_nx;
                n_nx = 0;
                if (e0 + 32 + lane < e1) { c_nx = hcls[e0 + 32 + lane]; n_nx = cb[c_nx]; }
                const bool take = n != 0;              // entries past the list end have n = 0
                const double t = take ? (double)n * (ph / z[c]) : 0.0;
                acc = add_in_lane_order(acc, t, take);
            }
            const double nw = acc / Td, d = fabs(nw - ph);
            wmax = wmax < d ? d : wmax;
            if (lane == 0) pi[h] = nw;                 // only this warp reads pi[h] in this phase
        }
        for (int o = 16; o; o >>= 1) {
            const double x = __shfl_xor_sync(FULL, wmax, o);
            wmax = wmax < x ? x : wmax;
        }
        if (lane == 0) s_max[warp] = wmax;
        __syncthreads();
        if (threadIdx.x == 0) {
            double m = 0.0;
            for (int w = 0; w < nwarps; ++w) m = m < s_max[w] ? s_max[w] : m;
            s_delta = m;
        }
        __syncthreads();
        delta = s_delta;
        if (delta <= tol) break;
    }
    // loglik: the terms count_c * log10(z_c) over the final pi, then one sum in class order
    for (int64_t c = threadIdx.x; c < C; c += blockDim.x) {
        const unsigned long long n = cb[c];
        if (!n) continue;
        double s = 0.0;
        for (int64_t j = class_off[c]; j < class_off[c + 1]; ++j) s += pi[members[j]];
        z[c] = (double)n * hx_gl_log10(s);
    }
    __syncthreads();
    if (warp == 0) {
        double ll = 0.0;
        for (int64_t c0 = 0; c0 < C; c0 += 32) {
            const int64_t c = c0 + lane;
            const bool take = c < C && cb[c];
            ll = add_in_lane_order(ll, take ? z[c] : 0.0, take);
        }
        if (lane == 0) {
            it_out[2 * r] = it;
            it_out[2 * r + 1] = delta <= tol;
            ll_out[r] = ll;
        }
    }
    if (in_smem)
        for (int h = threadIdx.x; h < H; h += blockDim.x) g_pi[(int64_t)r * H + h] = pi[h];
}

// replicates per batch: the scratch of one replicate is its counts, pi, n_iter + converged, loglik, and z when it
// does not fit in shared memory
int64_t boot_batch(int64_t H, int64_t C, bool in_smem) {
    const char *e = getenv("HX_BOOT_SCRATCH_MB");
    const double mb = e ? atof(e) : 256.0;
    const int64_t per = 8 * C + 8 * H + 16 + (in_smem ? 0 : 8 * C);
    return std::max<int64_t>(1, std::min<int64_t>(65535, (int64_t)(mb * 1048576.0 / per)));
}

}  // namespace

void hx_boot_free(hx_matrix *h) {
    cudaStream_t st = h->stream;
    h->bt_off.release(st); h->bt_cnt0.release(st); h->bt_pre.release(st); h->bt_hoff.release(st);
    h->bt_mem.release(st); h->bt_hcls.release(st); h->bt_it.release(st);
    h->bt_cnt.release(st); h->bt_pi.release(st); h->bt_z.release(st); h->bt_ll.release(st);
}

extern "C" int hx_em_bootstrap(hx_matrix *h, int32_t n_haps, int64_t n_classes, const int64_t *class_off,
                               const int32_t *members, const int64_t *count, int32_t n_boot, uint64_t seed,
                               int32_t max_iter, double tol, double *pi, int32_t *n_iter, int32_t *converged,
                               double *loglik, int64_t *boot_count) {
    HX_CHECK_ARG(h && n_haps >= 1 && n_classes >= 0 && n_boot >= 0 && max_iter >= 0 && tol >= 0.0 && pi && n_iter &&
                 converged && loglik);
    HX_CHECK_ARG(n_classes == 0 || (class_off && members && count));
    HX_CHECK_ARG(n_classes < INT32_MAX);
    int64_t T = 0;
    if (const int rc = hx_check_classes(n_haps, n_classes, class_off, members, count, &T)) return rc;
    const int64_t H = n_haps, C = n_classes, R = (int64_t)n_boot + 1, M = C ? class_off[C] : 0;
    h->use.last_ms[6] = h->use.last_ms[7] = 0.0f;
    if (T == 0) {                                    // no class: nothing to draw, every row is K7's T = 0 answer
        std::fill(pi, pi + R * H, 0.0);
        std::fill(n_iter, n_iter + R, 0);
        std::fill(converged, converged + R, 1);
        std::fill(loglik, loglik + R, 0.0);
        return HX_OK;
    }
    HX_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    for (int e = 0; e < 2; ++e)
        if (!h->a_ev[e]) HX_CUDA(cudaEventCreate(&h->a_ev[e]));

    // prefix sums of the counts, and each haplotype's member entries in class order
    std::vector<int64_t> pre(C + 1), hoff(H + 1, 0);
    std::vector<int32_t> hcls(M);
    for (int64_t c = 0; c < C; ++c) pre[c + 1] = pre[c] + count[c];
    for (int64_t j = 0; j < M; ++j) ++hoff[members[j] + 1];
    for (int64_t x = 0; x < H; ++x) hoff[x + 1] += hoff[x];
    std::vector<int64_t> cur(hoff.begin(), hoff.end() - 1);
    for (int64_t c = 0; c < C; ++c)
        for (int64_t j = class_off[c]; j < class_off[c + 1]; ++j) hcls[cur[members[j]]++] = (int32_t)c;

    HX_CUDA(h->bt_off.grow(8 * (C + 1), st));
    HX_CUDA(h->bt_mem.grow(4 * std::max<int64_t>(M, 1), st));
    HX_CUDA(h->bt_cnt0.grow(8 * C, st));
    HX_CUDA(h->bt_pre.grow(8 * (C + 1), st));
    HX_CUDA(h->bt_hoff.grow(8 * (H + 1), st));
    HX_CUDA(h->bt_hcls.grow(4 * std::max<int64_t>(M, 1), st));
    HX_CUDA(cudaMemcpyAsync(h->bt_off.p, class_off, 8 * (C + 1), cudaMemcpyHostToDevice, st));
    HX_CUDA(cudaMemcpyAsync(h->bt_mem.p, members, 4 * M, cudaMemcpyHostToDevice, st));
    HX_CUDA(cudaMemcpyAsync(h->bt_cnt0.p, count, 8 * C, cudaMemcpyHostToDevice, st));
    HX_CUDA(cudaMemcpyAsync(h->bt_pre.p, pre.data(), 8 * (C + 1), cudaMemcpyHostToDevice, st));
    HX_CUDA(cudaMemcpyAsync(h->bt_hoff.p, hoff.data(), 8 * (H + 1), cudaMemcpyHostToDevice, st));
    HX_CUDA(cudaMemcpyAsync(h->bt_hcls.p, hcls.data(), 4 * M, cudaMemcpyHostToDevice, st));

    const bool em_smem = 8 * (H + C) <= EM_SMEM_BYTES, draw_smem = C <= DRAW_SMEM_CLASSES;
    const size_t em_bytes = em_smem ? (size_t)(8 * (H + C)) : 0, draw_bytes = draw_smem ? (size_t)(12 * C + 8) : 0;
    HX_CUDA(cudaFuncSetAttribute(k_boot_em, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)em_bytes));
    HX_CUDA(cudaFuncSetAttribute(k_boot_draw<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)draw_bytes));
    const int64_t batch = std::min(R, boot_batch(H, C, em_smem));
    HX_CUDA(h->bt_cnt.grow(8 * batch * C, st));
    HX_CUDA(h->bt_pi.grow(8 * batch * H, st));
    HX_CUDA(h->bt_it.grow(8 * batch, st));
    HX_CUDA(h->bt_ll.grow(8 * batch, st));
    if (!em_smem) HX_CUDA(h->bt_z.grow(8 * batch * C, st));
    const uint64_t n_pairs = ((uint64_t)T + 1) / 2;
    const unsigned slices = (unsigned)((n_pairs + DRAW_PAIRS_PER_CTA - 1) / DRAW_PAIRS_PER_CTA);
    std::vector<int32_t> it_h(2 * batch);

    for (int64_t r0 = 0; r0 < R; r0 += batch) {
        const int64_t nb = std::min(batch, R - r0);
        HX_CUDA(hx_fill_async(h->bt_cnt.p, 0, 8 * nb * C, st));
        if (r0 == 0) HX_CUDA(cudaMemcpyAsync(h->bt_cnt.p, h->bt_cnt0.p, 8 * C, cudaMemcpyDeviceToDevice, st));
        const int64_t d0 = std::max<int64_t>(r0, 1), nd = r0 + nb - d0;   // replicates drawn in this batch
        int rc;
        if (nd > 0) {
            unsigned long long *rows = h->bt_cnt.p + (d0 - r0) * C;
            rc = timed(h, 6, [&] {
                const dim3 grid(slices, (unsigned)nd);
                if (draw_smem)
                    k_boot_draw<true><<<grid, DRAW_THREADS, draw_bytes, st>>>(h->bt_pre.p, C, (uint64_t)T, seed,
                                                                              (int)d0, rows);
                else
                    k_boot_draw<false><<<grid, DRAW_THREADS, 0, st>>>(h->bt_pre.p, C, (uint64_t)T, seed, (int)d0,
                                                                      rows);
            });
            if (rc) return rc;
        }
        rc = timed(h, 7, [&] {
            k_boot_em<<<(unsigned)nb, EM_THREADS, em_bytes, st>>>(
                (int)H, C, h->bt_off.p, h->bt_mem.p, h->bt_hoff.p, h->bt_hcls.p, h->bt_cnt.p, (double)T, max_iter, tol,
                em_smem, h->bt_pi.p, em_smem ? nullptr : h->bt_z.p, h->bt_it.p, h->bt_ll.p);
        });
        if (rc) return rc;
        HX_CUDA(cudaMemcpyAsync(pi + r0 * H, h->bt_pi.p, 8 * nb * H, cudaMemcpyDeviceToHost, st));
        HX_CUDA(cudaMemcpyAsync(loglik + r0, h->bt_ll.p, 8 * nb, cudaMemcpyDeviceToHost, st));
        HX_CUDA(cudaMemcpyAsync(it_h.data(), h->bt_it.p, 8 * nb, cudaMemcpyDeviceToHost, st));
        if (boot_count)
            HX_CUDA(cudaMemcpyAsync(boot_count + r0 * C, h->bt_cnt.p, 8 * nb * C, cudaMemcpyDeviceToHost, st));
        HX_CUDA(cudaStreamSynchronize(st));
        for (int64_t k = 0; k < nb; ++k) {
            n_iter[r0 + k] = it_h[2 * k];
            converged[r0 + k] = it_h[2 * k + 1];
        }
    }
    return HX_OK;
}
