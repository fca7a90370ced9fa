// Parity probe: an independent, deliberately simple recount of what every band row must hold, used by
// bench.py and the multi-GPU tests to check a finished ingestion (after the cross-GPU exchange) without a
// CPU oracle.  One thread per read walks its alleles once and adds, for every target site, the number of
// observations the pair-expansion rules of gretel/util.py:254-281 produce in that band row; the second
// kernel sums the counters the ingestion kernels actually wrote, row by row.  The two vectors must agree
// in every row (and their grand total must equal n_crumbs + sentinel increments).
#include "hx_internal.cuh"

namespace {

__device__ __forceinline__ bool probe_valid_from(unsigned a) {      // util.py:258
    return a != HX_SYM_N && a != HX_SYM_GAP && a <= 6;
}

__global__ void k_probe_expected_rows(const int32_t *__restrict__ rank, const int64_t *__restrict__ off,
                                      const uint8_t *__restrict__ codes, int64_t n_reads, int N, int W,
                                      unsigned long long *__restrict__ rows) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    const int64_t o = off[r];
    const int64_t k = off[r + 1] - o;
    if (k < 2) return;                                              // util.py:230
    const int rk = rank[r];
    if (rk < 0 || (int64_t)rk + k > N || k - 1 > W) return;         // the ingestion reports these as errors
    const uint8_t *c = codes + o;
    unsigned nvalid = probe_valid_from(c[0]);                       // valid first alleles among c[0..j-1]
    for (int64_t j = 1; j < k; ++j) {
        const unsigned b = c[j];
        if (b <= 6 && nvalid) atomicAdd(&rows[rk + j + 1], (unsigned long long)nvalid);
        nvalid += probe_valid_from(b);
    }
    if (rk == 0 && probe_valid_from(c[0]) && c[1] <= 6) atomicAdd(&rows[1], 1ull);             // :262-266
    if (rk + k == N && !(k == 2 && rk == 0) && probe_valid_from(c[k - 2]) && c[k - 1] <= 6)    // :271-275
        atomicAdd(&rows[N + 1], 1ull);
}

__global__ void k_counts_row_sums(const uint32_t *__restrict__ cnt, int64_t row_elems, int64_t n_rows,
                                  unsigned long long *__restrict__ rows) {
    const int64_t pj = blockIdx.x;
    if (pj >= n_rows) return;
    const uint32_t *p = cnt + pj * row_elems;
    unsigned long long s = 0;
    for (int64_t i = threadIdx.x; i < row_elems; i += blockDim.x) s += p[i];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ unsigned long long sh[32];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[w];
        rows[pj] = t;
    }
}

}  // namespace

extern "C" {

int hx_probe_expected_rows(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off, const uint8_t *d_codes,
                           int64_t n_reads, uint64_t *d_rows) {
    HX_CHECK_ARG(h && d_rows && n_reads >= 0);
    if (n_reads == 0) return HX_OK;
    HX_CHECK_ARG(d_rank && d_off && d_codes);
    HX_CUDA(cudaSetDevice(h->device));
    k_probe_expected_rows<<<(unsigned)((n_reads + 255) / 256), 256, 0, h->stream>>>(
        d_rank, d_off, d_codes, n_reads, h->N, h->W, reinterpret_cast<unsigned long long *>(d_rows));
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    return HX_OK;
}

int hx_counts_row_sums(hx_matrix *h, uint64_t *d_rows) {
    HX_CHECK_ARG(h && d_rows);
    if (!h->cnt) { hx_set_error("hx_counts_row_sums: no pending integer counts"); return HX_E_STATE; }
    HX_CUDA(cudaSetDevice(h->device));
    k_counts_row_sums<<<(unsigned)(h->N + 2), 256, 0, h->stream>>>(h->cnt, (int64_t)h->W * HX_CELL, (int64_t)h->N + 2,
                                                               reinterpret_cast<unsigned long long *>(d_rows));
    h->use.launches++;
    HX_CUDA(cudaGetLastError());
    return HX_OK;
}

}  // extern "C"
