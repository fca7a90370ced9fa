/* hanselx.h - C ABI of the B200-native Hansel matrix + Gretel recovery hot path.
 *
 * This is the drop-in boundary.  The reference has no FFI layer of its own: Gretel
 * is pure Python and reaches the matrix through the Python class ``hansel.Hansel``
 * (pip hanselx==0.0.92, /root/reference/setup.py:8) and three Python functions.
 * Each entry point below names the reference interface it stands behind
 * (paths relative to /root/reference).  INTEGRATION.md shows the ctypes binding a
 * Gretel maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary
 *   - every function returns an hx_status; HX_OK == 0, errors < 0, HX_HOLE > 0
 *   - hx_last_error() returns a thread-local message for the last failing call
 *   - host buffers are borrowed for the duration of the call only
 *   - symbols are codes 0..6 = A C G T N - _   (order fixed by gretel/util.py:83);
 *     unsymbols are N(4) and _(6)
 *   - positions: 0 = start sentinel, 1..N = SNP sites, N+1 = end sentinel
 *   - a read is (rank r >= 0, codes c[0..k-1]); c[t] is the allele at site r+t+1
 *
 * Storage: counts live in a diagonal band, cell (pi,pj) with 1 <= pj-pi <= W at
 * band[(pj*W + (pj-pi-1))*49 + a*7 + b].  Cells outside the band are structurally
 * zero for ingested reads as long as W >= (longest read's SNP count - 1).
 */
#ifndef HANSELX_H
#define HANSELX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hx_matrix hx_matrix;

typedef enum {
    HX_OK = 0,
    HX_HOLE = 1,        /* generate_path found no branch (gretel/gretel.py:176-180); not an error */
    HX_E_CUDA = -1,
    HX_E_ARG = -2,
    HX_E_BAND = -3,     /* cell outside the band */
    HX_E_READ = -4,     /* a packed read leaves [0,N], is wider than the band, or has a code > 6 */
    HX_E_NOMEM = -5,
    HX_E_STATE = -6
} hx_status;

/* flags for the recovery arithmetic (the switchable, unpinned choices; see oracle/) */
#define HX_F_VSITE_TO        1   /* Laplace denominator counts valid symbols at the *to* site */
#define HX_F_KEEP_UNSYMBOLS  2   /* offer N and _ as candidate branches */

const char *hx_last_error(void);
int hx_version(void);
int hx_device_count(int *n);

/* ---- lifetime ------------------------------------------------------------------- */
/* Hansel.init_matrix(symbols, unsymbols, N)            gretel/util.py:83 */
int hx_create(int32_t n_snps, int32_t band_w, int32_t device, hx_matrix **out);
int hx_destroy(hx_matrix *h);
/* Hansel.copy()                                        gretel/cmd.py:79 */
int hx_copy(const hx_matrix *src, hx_matrix **out);
int hx_info(const hx_matrix *h, int32_t *n_snps, int32_t *band_w, int32_t *device);
/* the CUDA stream all work of this matrix is ordered on (cudaStream_t as void*) */
int hx_stream(const hx_matrix *h, void **stream);
int hx_set_stream(hx_matrix *h, void *stream);
int hx_sync(hx_matrix *h);

/* ---- ingestion: replaces the pair-expansion loop gretel/util.py:226-286 --------- */
/* Host-buffer entry point (H2D + kernel + D2H of the totals), synchronous.
 * totals[4] = { n_slices (util.py:233), n_crumbs (util.py:268,276,281),
 *               covered_snps (util.py:239), sentinel increments }.
 * Counts accumulate over calls until hx_finalize_counts(). */
int hx_ingest_host(hx_matrix *h, const int32_t *rank, const int64_t *off, const uint8_t *codes,
                   int64_t n_reads, int64_t totals[4]);
/* The same, in the compact wire format (half the host->device bytes): klen[r] = SNPs on read r,
 * codes4 = the allele codes of all reads back to back, two per byte (low nibble first);
 * n_codes = sum of klen.  Offsets and byte codes are rebuilt on the device. */
int hx_ingest_host_compact(hx_matrix *h, const int32_t *rank, const uint16_t *klen, const uint8_t *codes4,
                           int64_t n_reads, int64_t n_codes, int64_t totals[4]);
/* The dense wire format for rank-sorted reads (about 6 bytes per 15-SNP read instead of 13.5): what the CPU
 * packer should emit for the GPU path.  See gretel_b200/csrc/wire.cu and gretel_b200.util.dense_packed.
 *   rank_delta uint8[n_reads]   rank[r]-rank[r-1] (rank[-1] = 0); 255 => the true delta is esc_delta[k] where
 *                               esc_idx[k] == r (esc_idx ascending; first read of a chunk, or a gap >= 255 sites)
 *   klen       uint8[n_reads] (klen_bytes = 1) or uint16[n_reads] (klen_bytes = 2): SNPs on read r
 *   codes2     2 bits per allele, four per byte, low bits first (A0 C1 G2 T3); N, '-' and '_' store code-4 and
 *              are listed, by index into the allele stream, in exc_pos[n_exc] (ascending)
 * totals != NULL: synchronous like hx_ingest_host.  totals == NULL: the call only enqueues (copies on a second
 * stream, rotating staging sets), so feeding the reads in a few chunks overlaps each copy with the previous chunk's
 * pair expansion; the host buffers must stay untouched until hx_ingest_totals() or hx_sync() returns. */
int hx_ingest_host_dense(hx_matrix *h, const uint8_t *rank_delta, const int64_t *esc_idx, const int32_t *esc_delta,
                         int64_t n_esc, const void *klen, int32_t klen_bytes, const uint8_t *codes2,
                         const uint32_t *exc_pos, int64_t n_exc, int64_t n_reads, int64_t n_codes,
                         int64_t totals[4]);
/* Device-buffer entry point, asynchronous on the matrix's stream. */
int hx_ingest_device(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off,
                     const uint8_t *d_codes, int64_t n_reads);
/* Select the ingestion kernel: 0 = auto, 1 = per-pair global reductions (generic),
 * 2 = bit-sliced shared-memory tiles (rank-sorted reads of <= 52 SNPs),
 * 3 = bit-plane transpose + owner-computes tiles (rank-sorted long reads),
 * 4 / 5 = force the barrier-phased / the warp-specialised variant of kernel 2 (2 picks by read width),
 * 6 = tensor-core kernel (int8 tcgen05.mma over one-hot allele rows; rank-sorted reads of <= 32 SNPs; what
 * auto picks for such reads),
 * 7 = long-read tensor-core kernel (counting sort of the reads by first/last site block, one-hot operand slabs,
 * int8 tcgen05.mma per 16 x 32-site tile; any read width, any order; what auto picks for reads wider than 52 SNPs). */
int hx_set_ingest_kernel(hx_matrix *h, int which);
/* Limit the persistent ingestion kernels to n_sms SMs (0 = all of them): leaves room for a collective that runs
 * beside the pair expansion of the next batch (bench.py --overlap-steps). */
int hx_set_ingest_sms(hx_matrix *h, int n_sms);
int hx_ingest_totals(hx_matrix *h, int64_t totals[4]);               /* synchronises */
/* Partial-matrix exchange across GPUs (the reference's fork-shared matrix,
 * util.py:303-326): device pointer + length of the uint32 counts and of the int64
 * totals, for an integer sum-allreduce by the caller (NCCL).  A caller that writes through the pointer
 * BEFORE an ingestion (rather than summing after it) must fetch it again after every hx_reset_counts: a
 * freshly cleared matrix lets the long-read kernel store instead of read-modify-write. */
int hx_counts_buffer(hx_matrix *h, void **d_counts, int64_t *n_u32, void **d_totals, int64_t *n_i64);
/* The same exchange with half the bytes: hx_counts_pack() copies the pending counts into a packed device
 * buffer (49 x uint16 per site pair in 25 words; the last 4 words are an overflow flag), the caller
 * sum-all-reduces its n_u32 uint32 words, and hx_counts_unpack() writes the sums back into the counts.  Lane
 * sums are exact when every count is <= 65535/world on every rank; otherwise *overflowed is 1, the counts are
 * untouched and the caller must fall back to hx_counts_buffer().  hx_counts_unpack synchronises. */
int hx_counts_pack(hx_matrix *h, int32_t world, void **d_packed, int64_t *n_u32);
int hx_counts_unpack(hx_matrix *h, int32_t *overflowed);
/* For exchanges that run behind the next ingestion (no host synchronisation per job): hx_counts_unpack_async launches
 * the write-back on `stream` (a cudaStream_t; NULL = the matrix's stream) and returns; hx_counts_pack_overflowed reads
 * the all-reduced overflow flag of the last packed exchange (synchronises).  hx_counts_max = the largest pending
 * count on this GPU (synchronises): packing is safe while max * world <= 65535. */
int hx_counts_unpack_async(hx_matrix *h, void *stream);
int hx_counts_pack_overflowed(hx_matrix *h, int32_t *overflowed);
int hx_counts_max(hx_matrix *h, uint32_t *max_count);
/* Fused exchange (one process per GPU, NVLink peer memory): band rows are dealt out to the ranks in
 * contiguous blocks of ceil((N+2)/world); after export + import every ingestion kernel adds its counts
 * straight into the GPU that owns the row, so when all ranks' kernels are done each rank holds the final
 * sums of its own rows and the partial matrices never have to be all-reduced (an all-gather of the owned
 * rows, or nothing if only the owner needs them, completes the exchange).
 *   hx_counts_ipc_export  (re)allocates the pending counts as an IPC-shareable buffer, padded to
 *                         world * rows_per rows, and writes its 64-byte cudaIpcMemHandle_t;
 *   hx_counts_ipc_import  takes the world handles (own one included, in rank order). */
int hx_counts_ipc_export(hx_matrix *h, int32_t world, void *handle_out);
int hx_counts_ipc_import(hx_matrix *h, const void *handles, int32_t world, int32_t my_rank);
/* Unmap the peers' buffers (every rank must do this before any rank frees its own: barrier around it). */
int hx_counts_ipc_close(hx_matrix *h);
/* Fold the integer counts into the float32 working matrix used by everything below
 * (util.py:329-333 happens in the caller from the totals). */
int hx_finalize_counts(hx_matrix *h);
/* Zero the pending integer counts and the totals (start a new ingestion job). */
int hx_reset_counts(hx_matrix *h);

/* ---- scalar Hansel surface ------------------------------------------------------- */
/* Hansel.add_observation(a,b,i,j)                      gretel/util.py:266-286 */
int hx_add_observation(hx_matrix *h, int a, int b, int32_t i, int32_t j, float amount);
/* Hansel.get_observation(a,b,i,j)                      tests/test_test.py:41-52 */
int hx_get_observation(hx_matrix *h, int a, int b, int32_t i, int32_t j, float *out);
/* Hansel.reweight_observation(a,b,i,j,ratio)->removed  gretel/gretel.py:84,96 */
int hx_reweight_observation(hx_matrix *h, int a, int b, int32_t i, int32_t j, double ratio,
                            double *removed);
/* Hansel.reweight_matrix(ratio)                        gretel/gretel.py:72 (dead code upstream) */
int hx_reweight_matrix(hx_matrix *h, double ratio);
/* Hansel.get_counts_at(i) for every i in 0..N          gretel/cmd.py:85-92,123-145
 * out[(N+1)*8]: 7 symbol counts (0 where absent) then the total. */
int hx_counts_all(hx_matrix *h, double *out);
/* Hansel.get_marginal_of_at(sym, pos)                  gretel/gretel.py:182,186 */
int hx_marginal_of_at(hx_matrix *h, int sym, int32_t pos, double *out);
/* Hansel.get_edge_weights_at(snp, path)                gretel/gretel.py:155
 * path[0..snp-1] are the symbols chosen so far (path[0] = '_').  weights[7] are the
 * normalised branch weights (0 where not a candidate), *mask the candidate set,
 * *total the "total" entry. */
int hx_edge_weights_at(hx_matrix *h, int32_t snp, const uint8_t *path, int32_t L, int flags,
                       double weights[7], double *total, int *mask);

/* ---- bulk recovery --------------------------------------------------------------- */
/* gretel.generate_path(n_snps, hansel, original_hansel) gretel/gretel.py:102-189
 * out_path[N+1]; out[3] = { hp_current, hp_original, min_marginal }.
 * Returns HX_HOLE with *hole_site = snp when no branch exists. */
int hx_generate_path(hx_matrix *cur, hx_matrix *orig, int32_t L, int flags, uint8_t *out_path,
                     double out[3], int32_t *hole_site);
/* gretel.reweight_hansel_from_path(hansel, path, ratio) gretel/gretel.py:13-98 */
int hx_reweight_path(hx_matrix *h, const uint8_t *path, double ratio, double *removed);
/* The recovery driver loop gretel/cmd.py:148-161 kept resident on the device:
 * up to max_paths x (generate_path; ratio = max(min_marginal, min_remove);
 * reweight).  paths[max_paths*(N+1)], stats[max_paths*5] = { hp_current,
 * hp_original, min_marginal, ratio, removed }.  *n_found = iterations completed. */
int hx_recover(hx_matrix *cur, hx_matrix *orig, int32_t L, int flags, int32_t max_paths,
               double min_remove, uint8_t *paths, double *stats, int32_t *n_found);

/* ---- read support ------------------------------------------------------------------ */
/* Read support for recovered haplotypes (no reference counterpart; see DESIGN.md).  haps[n_haps*(N+1)]: paths as
 * hx_recover writes them; reads as for hx_ingest_host (any order, any width).  max_mismatch < 0: no limit.
 * Per-haplotype unique/shared (int64) and share_q32 (uint64) [n_haps]; totals[3] = {assigned, uninformative,
 * over_limit}.  best_mm, n_best, first_best: int32[n_reads] each, or NULL.  Synchronous.
 * A read goes to the haplotypes with the fewest mismatches at its informative sites (codes other than N and _);
 * a tie splits it into floor(2^32/ties) per tied haplotype.  HX_E_READ: a read past site N or a code > 6;
 * HX_E_ARG: a haplotype code > 6 at a site in 1..N.  The matrix supplies N, the device, the stream and scratch;
 * its counts are neither read nor changed. */
int hx_assign_reads(hx_matrix *h, const uint8_t *haps, int32_t n_haps,
                    const int32_t *rank, const int64_t *off, const uint8_t *codes, int64_t n_reads,
                    int32_t max_mismatch, int64_t *unique, int64_t *shared, uint64_t *share_q32,
                    int64_t totals[3], int32_t *best_mm, int32_t *n_best, int32_t *first_best);

/* ---- path scores --------------------------------------------------------------------- */
/* Per-site branch weights of given haplotypes (no reference counterpart; DESIGN.md §4 K6).  haps[n_haps*(N+1)] as
 * hx_recover writes them.  Every per-site output is [n_haps*N] (site s of haplotype h at h*N + s-1) and may be NULL;
 * weights is [n_haps*N*8] (7 normalised weights, then the total) or NULL.  loglik, n_unsupported, n_disagree: [n_haps].
 * Site s of haplotype h gets exactly what hx_edge_weights_at(s, haps[h], L, flags) reports; best = the first maximum
 * over the candidates (255: none); w_hap = the weight of the haplotype's own allele (0 if it is not a candidate);
 * w_second = the largest weight of the other candidates (0 if none).  loglik = the sum of log10(w_hap) over the sites
 * with w_hap > 0 in site order; n_unsupported = the sites with w_hap = 0; n_disagree = the sites with best != the
 * haplotype's allele.  HX_E_ARG: a code > 6, or haps[h][0] != '_'.  The matrix's band and counts are not changed.
 * Synchronous. */
int hx_score_paths(hx_matrix *h, const uint8_t *haps, int32_t n_haps, int32_t L, int flags,
                   double *weights, double *w_hap, double *w_second, uint8_t *best,
                   double *loglik, int32_t *n_unsupported, int32_t *n_disagree);

/* ---- BAM -> packed reads on the CPU (the producer side of the boundary) ------------ */
/* Replaces the pysam column pileup of gretel/util.py:112-210: multi-threaded BGZF inflate and one
 * CIGAR walk per alignment against the sorted 1-based SNP positions.  stepper: 0 = samtools,
 * 1 = all, 2 = nofilter (gretel/cmd.py:39,78).  The arrays are malloc'ed; release with hx_pack_free. */
typedef struct {
    int32_t *rank;      /* [n_reads]   index of the first SNP on the read */
    int64_t *off;       /* [n_reads+1] */
    uint8_t *codes;     /* [n_codes]   A0 C1 G2 T3 N4 -5 */
    int64_t n_reads, n_codes, n_records;
} hx_packed;
int hx_pack_bam(const char *bam_path, const char *contig, int32_t start_pos, int32_t end_pos,
                const int32_t *snp_pos, int32_t n_snps, int stepper, int n_threads, hx_packed *out);
/* The same with pysam's pileup depth cap and stage timings.  max_depth > 0 reproduces bam_plp's buffer limit (the
 * reference never changes pysam's default of 8000, gretel/util.py:137): a read that is not the first of its start
 * position is dropped while max_depth reads are still buffered; 0 = keep every read.  stage_seconds (or NULL):
 * { file read, BGZF inflate, record scan, depth filter, CIGAR walks, gather }.  The BAM is streamed in bounded
 * waves of BGZF blocks and reading stops once a coordinate-sorted file has passed end_pos. */
int hx_pack_bam_ex(const char *bam_path, const char *contig, int32_t start_pos, int32_t end_pos,
                   const int32_t *snp_pos, int32_t n_snps, int stepper, int n_threads, int32_t max_depth,
                   hx_packed *out, double stage_seconds[6]);
void hx_pack_free(hx_packed *p);
/* Packed reads (rank-sorted) -> the dense wire format of hx_ingest_host_dense, as one malloc'ed buffer whose
 * sections sit at the given byte offsets (rank_delta at 0): shipping it takes a single host->device copy.
 * CPU code (n_threads workers).  HX_E_ARG if the reads are not sorted by rank.  Release with hx_dense_free. */
typedef struct hx_dense {
    uint8_t *blob;
    int64_t blob_bytes, n_reads, n_codes, n_exc, n_esc;
    int64_t o_klen, o_codes2, o_exc, o_esc_idx, o_esc_delta;
    int32_t klen_bytes;
} hx_dense;
int hx_dense_encode(const int32_t *rank, const int64_t *off, const uint8_t *codes, int64_t n_reads, int n_threads,
                    hx_dense *out);
void hx_dense_free(hx_dense *d);
/* Per-position A,C,G,T counts over 0-based [start0,end0) of a contig from every alignment, no filters:
 * what gretel/snpper.py:30 asks pysam.count_coverage for.  out[4*(end0-start0)], A row first. */
int hx_count_coverage(const char *bam_path, const char *contig, int32_t start0, int32_t end0, int n_threads,
                      uint32_t *out);
/* The same with the histogram on the GPU: the CPU decodes the BAM into aligned segments and 4-bit bases, a
 * shared-memory-privatised histogram kernel counts them (gretel/snpper.py:29-41).  out on the host. */
int hx_count_coverage_gpu(const char *bam_path, const char *contig, int32_t start0, int32_t end0, int n_threads,
                          int32_t device, uint32_t *out);
int hx_bam_contig_length(const char *bam_path, const char *contig, int32_t *length);
/* The packer's own raw-DEFLATE decoder (csrc/hx_inflate.h; what pysam/htslib's bgzf reader does with zlib under
 * gretel/util.py:137), exposed for the differential tests against zlib: src[0..n) inflates to exactly m bytes into dst;
 * n_readable >= n bytes of src may be read (a BGZF payload is followed by its 8-byte trailer).  use_zlib != 0 runs
 * zlib's inflate on the same buffers instead.  HX_OK or HX_E_ARG. */
int hx_inflate_raw(const uint8_t *src, int64_t n, int64_t n_readable, uint8_t *dst, int64_t m, int32_t use_zlib);

/* ---- parity probe (bench.py parity_probe, multi-GPU tests) ------------------------ */
/* An independent recount of gretel/util.py:254-281: adds into d_rows[N+2] (device, uint64) the number of
 * increments (observations + sentinel increments) the reads must leave in every band row pj.  Accumulates, so
 * several shards (or ranks, after an integer all-reduce of d_rows) can be summed. */
int hx_probe_expected_rows(hx_matrix *h, const int32_t *d_rank, const int64_t *d_off, const uint8_t *d_codes,
                           int64_t n_reads, uint64_t *d_rows);
/* Row sums of the pending integer counts (after any cross-GPU exchange): d_rows[N+2] (device, uint64). */
int hx_counts_row_sums(hx_matrix *h, uint64_t *d_rows);

/* ---- the recovery kernels' log10 / 10**x (diagnostic; tests) ------------------------ */
/* y[i] = log10(x[i]) (which = 0) or 10**x[i] (which = 1) evaluated ON THE DEVICE by the routines the recovery kernels
 * use: a transcription of glibc's log10() / pow() (what math.log10 and float ** reach at gretel/gretel.py:166-187),
 * bit-identical to the host's libm on this image.  x, y: host arrays of n doubles. */
int hx_device_math(int32_t device, int which, const double *x, double *y, int64_t n);

/* ---- bulk matrix I/O (tests, --dumpmatrix gretel/cmd.py:81-82) ------------------- */
int hx_band_to_host(hx_matrix *h, float *out /* (N+2)*W*49 */);
int hx_band_from_host(hx_matrix *h, const float *in);
int hx_to_dense(hx_matrix *h, float *out /* 7*7*(N+2)*(N+2) */);
/* last kernel timings in ms measured with CUDA events on the matrix's stream:
 * which = 0 ingest, 1 generate_path walk, 2 reweight, 3 the assignment kernels of the last hx_assign_reads
 * (copies excluded), 4 the scoring kernels of the last hx_score_paths (copies excluded) */
int hx_last_kernel_ms(hx_matrix *h, int which, float *ms);
/* number of kernel launches issued by this matrix so far */
int hx_launch_count(const hx_matrix *h, int64_t *n);

#ifdef __cplusplus
}
#endif
#endif /* HANSELX_H */
