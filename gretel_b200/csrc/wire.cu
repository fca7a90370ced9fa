// Dense wire format of rank-sorted packed reads: host -> device bytes are what bounds the end-to-end rate
// (PCIe), so the host side ships 1 byte of rank delta + 1 (or 2) bytes of SNP count per read and 2 bits per
// allele, and the device rebuilds the (rank int32, off int64, codes uint8) arrays the ingestion kernels read:
//
//   rank_delta uint8[R]   rank[r] - rank[r-1] (rank[-1] = 0); 255 => the true delta is listed in
//                         (esc_idx[], esc_delta[]) - first read of a chunk, or a gap of >= 255 SNP sites
//   klen       uint8[R] | uint16[R]   SNPs on read r
//   codes2     2 bits per allele, four per byte, low bits first: A0 C1 G2 T3; an allele that is N, '-' or '_'
//              stores code-4 and its index in the allele stream is listed in exc_pos[] (ascending uint32)
//
// One pass of partial sums, a spine and an apply pass yield both scans (ranks inclusive, offsets exclusive).
// hx_ingest_host_dense(..., totals = NULL) only enqueues: copies go on a second stream into one of three staging
// sets and the decode on a third, so the copy and decode of chunk i+1 overlap the pair expansion of chunk i.
#include <algorithm>
#include <stdlib.h>
#include <thread>

#include "dense_enc.h"
#include "hx_internal.cuh"

namespace {

constexpr int WI = 16;                     // reads per thread
constexpr int WB = 256 * WI;               // reads per block

__device__ __forceinline__ int32_t esc_lookup(const int64_t *__restrict__ idx, const int32_t *__restrict__ delta,
                                              int64_t n_esc, int64_t j) {
    int64_t lo = 0, hi = n_esc;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (idx[mid] < j) lo = mid + 1; else hi = mid;
    }
    return lo < n_esc && idx[lo] == j ? delta[lo] : 255;
}

// 16 consecutive reads of one thread: rank deltas and SNP counts (zero beyond n)
template <int KB>
__device__ __forceinline__ void load_reads(const uint8_t *__restrict__ rd, const void *__restrict__ kl, int64_t j0,
                                           int64_t n, const int64_t *__restrict__ esc_idx,
                                           const int32_t *__restrict__ esc_delta, int64_t n_esc, int32_t (&d)[WI],
                                           int32_t (&k)[WI]) {
    if (j0 + WI <= n) {
        const uint4 a = *reinterpret_cast<const uint4 *>(rd + j0);
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int i = 0; i < WI; ++i) d[i] = (int32_t)((aw[i >> 2] >> (8 * (i & 3))) & 0xffu);
        if (KB == 1) {
            const uint4 b = *reinterpret_cast<const uint4 *>(static_cast<const uint8_t *>(kl) + j0);
            const uint32_t bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < WI; ++i) k[i] = (int32_t)((bw[i >> 2] >> (8 * (i & 3))) & 0xffu);
        } else {
            const uint4 *p = reinterpret_cast<const uint4 *>(static_cast<const uint16_t *>(kl) + j0);
            const uint4 b0 = p[0], b1 = p[1];
            const uint32_t bw[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < WI; ++i) k[i] = (int32_t)((bw[i >> 1] >> (16 * (i & 1))) & 0xffffu);
        }
    } else {
#pragma unroll
        for (int i = 0; i < WI; ++i) {
            const int64_t j = j0 + i;
            d[i] = j < n ? (int32_t)rd[j] : 0;
            k[i] = j < n ? (KB == 1 ? (int32_t)static_cast<const uint8_t *>(kl)[j]
                                    : (int32_t)static_cast<const uint16_t *>(kl)[j])
                         : 0;
        }
    }
    if (n_esc) {
#pragma unroll
        for (int i = 0; i < WI; ++i)
            if (d[i] == 255) {
                const int32_t e = esc_lookup(esc_idx, esc_delta, n_esc, j0 + i);
                d[i] = e < 0 ? 0 : e;              // ranks must never decrease: the expansion relies on it
            }
    }
}

template <int KB>
__global__ void __launch_bounds__(256)
k_dense_partials(const uint8_t *__restrict__ rd, const void *__restrict__ kl, int64_t n,
                 const int64_t *__restrict__ esc_idx, const int32_t *__restrict__ esc_delta, int64_t n_esc,
                 int64_t *__restrict__ partials /* [2*nblk] */) {
    __shared__ int64_t sh[2][8];
    int32_t d[WI], k[WI];
    load_reads<KB>(rd, kl, (int64_t)blockIdx.x * WB + (int64_t)threadIdx.x * WI, n, esc_idx, esc_delta, n_esc, d, k);
    int64_t sd = 0, sk = 0;
#pragma unroll
    for (int i = 0; i < WI; ++i) { sd += d[i]; sk += k[i]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sd += __shfl_xor_sync(0xffffffffu, sd, o);
        sk += __shfl_xor_sync(0xffffffffu, sk, o);
    }
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = sd; sh[1][threadIdx.x >> 5] = sk; }
    __syncthreads();
    if (threadIdx.x < 2) {
        int64_t t = 0;
        for (int w = 0; w < 8; ++w) t += sh[threadIdx.x][w];
        partials[2 * (int64_t)blockIdx.x + threadIdx.x] = t;
    }
}

// exclusive scan of the block partials: one CTA, 1024 blocks per step
// ... and the consistency check of the chunk: the SNP counts must add up to the allele count the caller stated
// (otherwise offsets would run past the unpacked codes).  *ok gates the pair expansion of this chunk.
__global__ void __launch_bounds__(1024) k_dense_spine(int64_t *__restrict__ partials, int64_t nblk, int64_t n_codes,
                                                      int *__restrict__ ok, int *__restrict__ err) {
    __shared__ int64_t sh[2][32];
    __shared__ int64_t carry[2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 2) carry[threadIdx.x] = 0;
    __syncthreads();
    for (int64_t b0 = 0; b0 < nblk; b0 += 1024) {
        const int64_t b = b0 + threadIdx.x;
        const int64_t vd = b < nblk ? partials[2 * b] : 0, vk = b < nblk ? partials[2 * b + 1] : 0;
        int64_t sd = vd, sk = vk;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t td = __shfl_up_sync(0xffffffffu, sd, o), tk = __shfl_up_sync(0xffffffffu, sk, o);
            if (lane >= o) { sd += td; sk += tk; }
        }
        if (lane == 31) { sh[0][warp] = sd; sh[1][warp] = sk; }
        __syncthreads();
        if (warp == 0) {                                  // scan of the 32 warp totals
            int64_t wd = sh[0][lane], wk = sh[1][lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t td = __shfl_up_sync(0xffffffffu, wd, o), tk = __shfl_up_sync(0xffffffffu, wk, o);
                if (lane >= o) { wd += td; wk += tk; }
            }
            sh[0][lane] = wd;
            sh[1][lane] = wk;
        }
        __syncthreads();
        const int64_t base_d = carry[0] + (warp ? sh[0][warp - 1] : 0), base_k = carry[1] + (warp ? sh[1][warp - 1] : 0);
        if (b < nblk) { partials[2 * b] = base_d + sd - vd; partials[2 * b + 1] = base_k + sk - vk; }
        __syncthreads();
        if (threadIdx.x == 0) { carry[0] += sh[0][31]; carry[1] += sh[1][31]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const bool good = carry[1] == n_codes;
        *ok = good ? 1 : 0;
        if (!good) atomicOr(err, 1);
    }
}

template <int KB>
__global__ void __launch_bounds__(256)
k_dense_apply(const uint8_t *__restrict__ rd, const void *__restrict__ kl, int64_t n,
              const int64_t *__restrict__ esc_idx, const int32_t *__restrict__ esc_delta, int64_t n_esc,
              const int64_t *__restrict__ partials, int32_t *__restrict__ rank, int64_t *__restrict__ off /* n+1 */,
              int N, int64_t *__restrict__ run_end) {
    __shared__ int64_t sh[2][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t j0 = (int64_t)blockIdx.x * WB + (int64_t)threadIdx.x * WI;
    int32_t d[WI], k[WI];
    load_reads<KB>(rd, kl, j0, n, esc_idx, esc_delta, n_esc, d, k);
    int64_t sd = 0, sk = 0;
#pragma unroll
    for (int i = 0; i < WI; ++i) { sd += d[i]; sk += k[i]; }
    int64_t id = sd, ik = sk;                        // inclusive scans over the warp's thread sums
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t td = __shfl_up_sync(0xffffffffu, id, o), tk = __shfl_up_sync(0xffffffffu, ik, o);
        if (lane >= o) { id += td; ik += tk; }
    }
    if (lane == 31) { sh[0][warp] = id; sh[1][warp] = ik; }
    __syncthreads();
    int64_t run_d = partials[2 * (int64_t)blockIdx.x] + id - sd;
    int64_t run_k = partials[2 * (int64_t)blockIdx.x + 1] + ik - sk;
    for (int w = 0; w < warp; ++w) { run_d += sh[0][w]; run_k += sh[1][w]; }
    // the delta of the read after this thread's 16: run_end[r] = index after the last read of rank r (what
    // k_prepass of ingest.cu records), so the pair expansion needs no pass of its own over the ranks
    int32_t d_next = 0;
    if (j0 + WI < n) {
        d_next = (int32_t)rd[j0 + WI];
        if (n_esc && d_next == 255) {
            d_next = esc_lookup(esc_idx, esc_delta, n_esc, j0 + WI);
            if (d_next < 0) d_next = 0;
        }
    }
#pragma unroll
    for (int i = 0; i < WI; ++i) {
        const int64_t j = j0 + i;
        run_d += d[i];
        if (j < n) {
            rank[j] = (int32_t)(run_d <= (int64_t)N + 1 ? run_d : (int64_t)N + 1);   // > N is invalid anyway; stays monotonic
            const int32_t dn = i + 1 < WI ? d[i + 1] : d_next;          // d[] is 0 beyond n
            if ((j + 1 == n || dn != 0) && run_d <= N) run_end[run_d] = j + 1;
        }
        if (j <= n) off[j] = run_k;
        run_k += k[i];
    }
}

// 16 alleles per thread: 2-bit fields -> bytes
__global__ void k_unpack_2bit(const uint32_t *__restrict__ in, int64_t n_words, uint4 *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words) return;
    const uint32_t w = in[i];
    uint32_t o[4];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        uint32_t x = (w >> (8 * b)) & 0xffu;
        x = (x | (x << 12)) & 0x000f000fu;
        o[b] = (x | (x << 6)) & 0x03030303u;
    }
    out[i] = make_uint4(o[0], o[1], o[2], o[3]);
}

__global__ void k_patch_exceptions(const uint32_t *__restrict__ pos, int64_t n_exc, int64_t n_codes,
                                   uint8_t *__restrict__ codes, int *__restrict__ err) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_exc) return;
    const uint32_t p = pos[i];
    if ((int64_t)p >= n_codes) { atomicOr(err, 2); return; }
    codes[p] = (uint8_t)(codes[p] + 4);              // N/-/_ were shipped as code-4 (a field value of 3 -> 7 is flagged later)
}

inline int64_t al16(int64_t x) { return (x + 15) & ~(int64_t)15; }

// HX_WIRE_TRACE=1: time every chunk's copy / decode / expansion on their streams and print the timeline at the
// next hx_ingest_totals() (debugging aid for the copy/compute overlap)
struct WireTrace {
    static constexpr int MAXC = 32;
    cudaEvent_t ev[MAXC][5];
    int64_t bytes[MAXC];
    int n = 0;
    bool made = false;
};
WireTrace g_trace;
const bool g_trace_on = getenv("HX_WIRE_TRACE") != nullptr;
void trace_mark(int which, cudaStream_t s) {
    if (!g_trace_on || g_trace.n >= WireTrace::MAXC) return;
    if (!g_trace.made) {
        for (auto &row : g_trace.ev) for (auto &e : row) cudaEventCreate(&e);
        g_trace.made = true;
    }
    cudaEventRecord(g_trace.ev[g_trace.n][which], s);
}

}  // namespace

void hx_wire_trace_dump() {
    if (!g_trace_on || g_trace.n == 0) return;
    cudaEventSynchronize(g_trace.ev[g_trace.n - 1][3]);
    for (int c = 0; c < g_trace.n; ++c) {
        float t[5];
        for (int i = 0; i < 5; ++i) cudaEventElapsedTime(&t[i], g_trace.ev[0][0], g_trace.ev[c][i]);
        fprintf(stderr, "[wire] chunk %d: copy %.3f..%.3f ms (%.1f GB/s)  decode ..%.3f  expand %.3f..%.3f\n", c, t[0], t[1],
                g_trace.bytes[c] / ((t[1] - t[0]) * 1e6), t[2], t[4], t[3]);
    }
    g_trace.n = 0;
}

void hx_wire_free(hx_matrix *h) {
    for (int s = 0; s < HX_WIRE_SETS; ++s) {
        hx_wire_set &w = h->wire[s];
        w.raw.release(h->stream); w.rank.release(h->stream); w.off.release(h->stream);
        w.codes.release(h->stream); w.partials.release(h->stream); w.run_end.release(h->stream);
        if (w.copied) cudaEventDestroy(w.copied);
        if (w.consumed) cudaEventDestroy(w.consumed);
        if (w.decoded) cudaEventDestroy(w.decoded);
        w = hx_wire_set{};
    }
    for (int s = 0; s < 2; ++s) {
        if (h->pin_ev[s]) cudaEventDestroy(h->pin_ev[s]);
        if (h->pin[s]) cudaFreeHost(h->pin[s]);
        h->pin[s] = nullptr; h->pin_cap[s] = 0; h->pin_ev[s] = nullptr; h->pin_busy[s] = false;
    }
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->decode_stream) cudaStreamDestroy(h->decode_stream);
    h->copy_stream = nullptr;
    h->decode_stream = nullptr;
}

// raw_codes != NULL: the "slim" variant - the allele bytes are copied as they are (from the caller's memory, before
// the small encoded sections), codes2 / exc_pos are unused
static int ingest_dense_impl(hx_matrix *h, const uint8_t *rank_delta, const int64_t *esc_idx,
                             const int32_t *esc_delta, int64_t n_esc, const void *klen, int32_t klen_bytes,
                             const uint8_t *codes2, const uint32_t *exc_pos, int64_t n_exc, int64_t n_reads,
                             int64_t n_codes, int64_t totals[4], const uint8_t *raw_codes) {
    HX_CHECK_ARG(h && n_reads >= 0 && n_codes >= 0 && n_esc >= 0 && n_exc >= 0);
    HX_CHECK_ARG(klen_bytes == 1 || klen_bytes == 2);
    HX_CHECK_ARG(n_codes < ((int64_t)1 << 32));
    HX_CUDA(cudaSetDevice(h->device));
    if (n_reads > 0) {
        HX_CHECK_ARG(rank_delta && klen && (codes2 || raw_codes || n_codes == 0) && (exc_pos || n_exc == 0));
        HX_CHECK_ARG(n_esc == 0 || (esc_idx && esc_delta));
        cudaStream_t st = h->stream;
        if (!h->copy_stream) HX_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        if (!h->decode_stream) HX_CUDA(cudaStreamCreateWithFlags(&h->decode_stream, cudaStreamNonBlocking));
        cudaStream_t ds = h->decode_stream;
        hx_wire_set &w = h->wire[h->use.wire_next];
        h->use.wire_next = (h->use.wire_next + 1) % HX_WIRE_SETS;
        const int64_t n_words = (n_codes + 15) / 16;        // 32-bit words of 2-bit alleles
        const int64_t n_words_sent = raw_codes ? 0 : n_words;
        const int64_t o_rd = 0, o_kl = o_rd + al16(n_reads), o_c2 = o_kl + al16(n_reads * klen_bytes);
        const int64_t o_ex = o_c2 + al16(n_words_sent * 4), o_ei = o_ex + al16(n_exc * 4), o_ed = o_ei + al16(n_esc * 8);
        const int64_t raw_bytes = o_ed + al16(n_esc * 4) + 16;
        const int64_t nblk = (n_reads + 1 + WB - 1) / WB;
        // `consumed` was recorded after the previous use of a staging set: the copy stream may overwrite the set
        // once that chunk's kernels are done, while the other sets' chunks are still being expanded.  All sets
        // are sized together (with headroom, chunks are about equal) so that a (re)allocation - which is ordered
        // on the compute stream and therefore moves the event to "now" - happens on the first chunk only.
        for (int s2 = 0; s2 < HX_WIRE_SETS; ++s2) {
            hx_wire_set &ws = h->wire[s2];
            if (!ws.copied) {
                HX_CUDA(cudaEventCreateWithFlags(&ws.copied, cudaEventDisableTiming));
                HX_CUDA(cudaEventCreateWithFlags(&ws.consumed, cudaEventDisableTiming));
                HX_CUDA(cudaEventCreateWithFlags(&ws.decoded, cudaEventDisableTiming));
            }
            bool grew = false;
            // a buffer too small for `need` bytes grows to `need` plus headroom
            auto fit = [&](auto &buf, int64_t need) {
                return need > buf.cap ? buf.grow(need + need / 8 + 256, st, &grew) : cudaSuccess;
            };
            HX_CUDA(fit(ws.raw, raw_bytes));
            HX_CUDA(fit(ws.rank, 4 * n_reads + 16));
            HX_CUDA(fit(ws.off, 8 * (n_reads + 1) + 16));
            HX_CUDA(fit(ws.codes, n_words * 16 + 32));
            HX_CUDA(fit(ws.partials, 16 * nblk + 32));
            HX_CUDA(ws.run_end.grow(8 * ((int64_t)h->N + 2), st, &grew));
            if (grew) HX_CUDA(cudaEventRecord(ws.consumed, st));
        }
        cudaStream_t cs = h->copy_stream;
        HX_CUDA(cudaStreamWaitEvent(cs, w.consumed, 0));
        trace_mark(0, cs);
        uint8_t *raw = w.raw.p;
        // util.dense_packed lays the arrays out in one host buffer exactly like the staging set: one copy
        const uint8_t *hb = rank_delta;
        if (raw_codes && n_codes) HX_CUDA(cudaMemcpyAsync(w.codes.p, raw_codes, (size_t)n_codes, cudaMemcpyHostToDevice, cs));
        const bool blob = (const uint8_t *)klen == hb + o_kl && (n_codes == 0 || raw_codes || codes2 == hb + o_c2) &&
                          (n_exc == 0 || (const uint8_t *)exc_pos == hb + o_ex) &&
                          (n_esc == 0 || ((const uint8_t *)esc_idx == hb + o_ei && (const uint8_t *)esc_delta == hb + o_ed));
        if (blob) {
            const int64_t used = n_esc ? o_ed + n_esc * 4 : (n_exc ? o_ex + n_exc * 4 : (n_codes && !raw_codes ? o_c2 + (n_codes + 3) / 4
                                                                                        : o_kl + n_reads * klen_bytes));
            HX_CUDA(cudaMemcpyAsync(raw, hb, (size_t)used, cudaMemcpyHostToDevice, cs));
        } else {
        HX_CUDA(cudaMemcpyAsync(raw + o_rd, rank_delta, (size_t)n_reads, cudaMemcpyHostToDevice, cs));
        HX_CUDA(cudaMemcpyAsync(raw + o_kl, klen, (size_t)(n_reads * klen_bytes), cudaMemcpyHostToDevice, cs));
        if (n_esc) {
            HX_CUDA(cudaMemcpyAsync(raw + o_ei, esc_idx, (size_t)(n_esc * 8), cudaMemcpyHostToDevice, cs));
            HX_CUDA(cudaMemcpyAsync(raw + o_ed, esc_delta, (size_t)(n_esc * 4), cudaMemcpyHostToDevice, cs));
        }
        if (n_codes && !raw_codes) HX_CUDA(cudaMemcpyAsync(raw + o_c2, codes2, (size_t)((n_codes + 3) / 4), cudaMemcpyHostToDevice, cs));
        if (n_exc) HX_CUDA(cudaMemcpyAsync(raw + o_ex, exc_pos, (size_t)(n_exc * 4), cudaMemcpyHostToDevice, cs));
        }
        trace_mark(1, cs);
        HX_CUDA(cudaEventRecord(w.copied, cs));
        // the decode runs on its own stream: it overlaps the previous chunk's expansion and the next chunk's copy
        HX_CUDA(cudaStreamWaitEvent(ds, w.copied, 0));
        int *ok = reinterpret_cast<int *>(w.partials.p + 2 * nblk);        // behind the block partials
        const int64_t *d_ei = reinterpret_cast<const int64_t *>(raw + o_ei);
        const int32_t *d_ed = reinterpret_cast<const int32_t *>(raw + o_ed);
        HX_CUDA(hx_fill_async(w.run_end.p, 0xff, sizeof(int64_t) * ((size_t)h->N + 2), ds));   // -1 = rank without reads
        h->use.launches++;
        if (klen_bytes == 1) {
            k_dense_partials<1><<<(unsigned)nblk, 256, 0, ds>>>(raw + o_rd, raw + o_kl, n_reads, d_ei, d_ed, n_esc, w.partials.p);
            k_dense_spine<<<1, 1024, 0, ds>>>(w.partials.p, nblk, n_codes, ok, h->d_err.p);
            k_dense_apply<1><<<(unsigned)nblk, 256, 0, ds>>>(raw + o_rd, raw + o_kl, n_reads, d_ei, d_ed, n_esc, w.partials.p,
                                                            w.rank.p, w.off.p, h->N, w.run_end.p);
        } else {
            k_dense_partials<2><<<(unsigned)nblk, 256, 0, ds>>>(raw + o_rd, raw + o_kl, n_reads, d_ei, d_ed, n_esc, w.partials.p);
            k_dense_spine<<<1, 1024, 0, ds>>>(w.partials.p, nblk, n_codes, ok, h->d_err.p);
            k_dense_apply<2><<<(unsigned)nblk, 256, 0, ds>>>(raw + o_rd, raw + o_kl, n_reads, d_ei, d_ed, n_esc, w.partials.p,
                                                            w.rank.p, w.off.p, h->N, w.run_end.p);
        }
        h->use.launches += 3;
        if (n_words_sent) {
            k_unpack_2bit<<<(unsigned)((n_words + 255) / 256), 256, 0, ds>>>(reinterpret_cast<const uint32_t *>(raw + o_c2),
                                                                            n_words, reinterpret_cast<uint4 *>(w.codes.p));
            h->use.launches++;
        }
        if (n_exc) {
            k_patch_exceptions<<<(unsigned)((n_exc + 255) / 256), 256, 0, ds>>>(
                reinterpret_cast<const uint32_t *>(raw + o_ex), n_exc, n_codes, w.codes.p, h->d_err.p);
            h->use.launches++;
        }
        HX_CUDA(cudaGetLastError());
        trace_mark(2, ds);
        HX_CUDA(cudaEventRecord(w.decoded, ds));
        HX_CUDA(cudaStreamWaitEvent(st, w.decoded, 0));
        int rc = hx_ensure_counts_buffer(h);
        if (rc) return rc;
        trace_mark(4, st);
        rc = hx_launch_ingest_presorted(h, w.rank.p, w.off.p, w.codes.p, n_reads, w.run_end.p, ok);
        if (rc) return rc;
        trace_mark(3, st);
        if (g_trace_on && g_trace.n < WireTrace::MAXC) g_trace.bytes[g_trace.n++] = raw_bytes;
        HX_CUDA(cudaEventRecord(w.consumed, st));
    }
    return totals ? hx_ingest_totals(h, totals) : HX_OK;
}

extern "C" int hx_ingest_host_dense(hx_matrix *h, const uint8_t *rank_delta, const int64_t *esc_idx,
                                    const int32_t *esc_delta, int64_t n_esc, const void *klen, int32_t klen_bytes,
                                    const uint8_t *codes2, const uint32_t *exc_pos, int64_t n_exc, int64_t n_reads,
                                    int64_t n_codes, int64_t totals[4]) {
    return ingest_dense_impl(h, rank_delta, esc_idx, esc_delta, n_esc, klen, klen_bytes, codes2, exc_pos, n_exc, n_reads,
                             n_codes, totals, nullptr);
}


// ---- host arrays -> matrix, pipelined -------------------------------------------------------------------------
// hx_ingest_host for large rank-sorted inputs: the packed arrays are cut into a few chunks at read boundaries;
// each chunk is encoded into the dense wire format by the host threads straight into one of two pinned buffers
// and enqueued with hx_ingest_host_dense(totals = NULL), so the encoding of chunk i+1 runs while chunk i is
// copied, decoded and pair-expanded.  HX_E_STATE = the reads are not sorted by rank (the caller ships them as
// they are) from read *done_reads on; the reads before it have been enqueued.
int hx_ingest_host_pipelined(hx_matrix *h, const int32_t *rank, const int64_t *off, const uint8_t *codes, int64_t n_reads,
                             bool slim, int64_t *done_reads) {
    *done_reads = 0;
    int nt = 0;
    if (const char *e = getenv("HX_HOST_THREADS")) nt = atoi(e);
    if (nt <= 0) nt = (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency()));
    const int64_t n_codes = off[n_reads] - off[0];
    constexpr int64_t CHUNK_CODES = (int64_t)32 << 20;
    int n_chunks = (int)std::max<int64_t>(slim ? 6 : 3, (n_codes + CHUNK_CODES - 1) / CHUNK_CODES);
    if (slim && nt > 8) nt = 8;                       // a few hundred microseconds of work per chunk
    if ((int64_t)n_chunks > n_reads) n_chunks = (int)n_reads;
    int64_t a = 0;
    static thread_local HxDensePlan plan;             // keeps its list buffers between chunks and calls
    for (int c = 0; c < n_chunks; ++c) {
        const int64_t b = hx_chunk_end(off, a, n_reads, n_codes, c, n_chunks);
        if (b <= a && c + 1 < n_chunks) continue;
        HxDensePlan &P = plan;
        int rc = hx_dense_begin(off + a, b - a, nt, (int64_t)h->W + 1, &P, slim);
        if (rc) return rc;
        const int slot = c & 1;
        if (h->pin_busy[slot]) { HX_CUDA(cudaEventSynchronize(h->pin_ev[slot])); h->pin_busy[slot] = false; }
        auto ensure_pin = [&](int64_t bytes, int64_t keep) -> int {
            if (bytes <= h->pin_cap[slot]) return HX_OK;
            const int64_t want = bytes + bytes / 8 + ((int64_t)1 << 20);
            uint8_t *np = nullptr;
            HX_CUDA(cudaHostAlloc((void **)&np, (size_t)want, cudaHostAllocPortable));
            if (keep > 0) memcpy(np, h->pin[slot], (size_t)keep);
            if (h->pin[slot]) cudaFreeHost(h->pin[slot]);
            h->pin[slot] = np;
            h->pin_cap[slot] = want;
            return HX_OK;
        };
        rc = ensure_pin(P.head_bytes + 16, 0);
        if (rc) return rc;
        if (!h->pin_ev[slot]) HX_CUDA(cudaEventCreateWithFlags(&h->pin_ev[slot], cudaEventDisableTiming));
        rc = hx_dense_pack(rank + a, off + a, codes, &P, h->pin[slot]);
        if (rc) return rc;                         // HX_E_STATE: not sorted from here on; *done_reads went out already
        rc = ensure_pin(P.bytes, P.head_bytes);
        if (rc) return rc;
        uint8_t *blob = h->pin[slot];
        hx_dense_finish(&P, blob);
        rc = ingest_dense_impl(h, blob, reinterpret_cast<const int64_t *>(blob + P.o_esc_idx),
                               reinterpret_cast<const int32_t *>(blob + P.o_esc_delta), P.n_esc, blob + P.o_klen,
                               P.klen_bytes, blob + P.o_codes2, reinterpret_cast<const uint32_t *>(blob + P.o_exc), P.n_exc,
                               b - a, P.n_codes, nullptr, slim ? codes + off[a] : nullptr);
        if (rc) return rc;
        HX_CUDA(cudaEventRecord(h->pin_ev[slot], h->copy_stream));      // the slot is free again once its copy is done
        h->pin_busy[slot] = true;
        a = b;
        *done_reads = a;
    }
    return HX_OK;
}
