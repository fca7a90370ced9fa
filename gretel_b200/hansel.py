"""Drop-in ``Hansel`` backed by the device-resident banded matrix of libhanselx.so.

Mirrors the surface of ``hansel.Hansel`` (pip hanselx==0.0.92, /root/reference/setup.py:8)
that Gretel uses: init_matrix (util.py:83), add_observation (util.py:266-286),
get_observation (tests/test_test.py:41-52), get_counts_at (cmd.py:86,127),
get_edge_weights_at (gretel.py:155), get_marginal_of_at (gretel.py:182,186),
reweight_observation (gretel.py:84,96), reweight_matrix (gretel.py:72), copy (cmd.py:79),
save_hansel_dump (cmd.py:82), attributes symbols_d / L / n_slices / n_crumbs.

Symbols are plain ``str`` (every use in Gretel - str(x), ==, dict key - is satisfied).
All arithmetic runs in CUDA kernels; there is no CPU fallback.  Cells outside the
diagonal band (j-i < 1 or j-i > band_w) can still be set through the scalar API - they
live in a small host-side spill dict and never take part in recovery, exactly as a
structurally-zero cell would for ingested reads.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib

REF_SYMBOLS = ['A', 'C', 'G', 'T', 'N', '-', '_']       # util.py:83
REF_UNSYMBOLS = ['N', '_']
_DENSE_BAND_LIMIT_BYTES = 2 << 30


def _default_device():
    return int(os.environ.get("GRETEL_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))


class ReadSupport:
    """What Hansel.assign_reads reports.  Per haplotype: ``unique`` (reads whose only best haplotype it is),
    ``shared`` (reads tied between it and others), ``share_q32`` (uint64: the sum of floor(2^32/ties) over the
    reads it is a best haplotype of) and ``share`` = share_q32 / 2^32.  Totals ``assigned``, ``uninformative``
    (no informative site) and ``over_limit`` (fewest mismatches above max_mismatch).  With per_read: ``best_mm``
    (fewest mismatches, -1 if uninformative), ``n_best`` (ties, 0 if uninformative), ``first_best`` (lowest best
    haplotype, -1 unless assigned); None otherwise."""

    def __init__(self, unique, shared, share_q32, assigned, uninformative, over_limit, best_mm=None, n_best=None,
                 first_best=None):
        self.unique, self.shared, self.share_q32 = unique, shared, share_q32
        self.share = share_q32.astype(np.float64) / 2.0 ** 32
        self.assigned, self.uninformative, self.over_limit = assigned, uninformative, over_limit
        self.best_mm, self.n_best, self.first_best = best_mm, n_best, first_best


class ReadClasses:
    """What Hansel.read_classes reports: the compatibility classes of the assigned reads (DESIGN.md §4 K7) as CSR.
    Class c has the haplotypes ``members[class_off[c]:class_off[c+1]]`` (int32, ascending), the tie set of its
    reads, and ``count[c]`` reads (int64, >= 1); classes are ordered lexicographically by member list.  Totals
    ``assigned`` (the sum of ``count``), ``uninformative`` and ``over_limit`` as in ReadSupport."""

    def __init__(self, class_off, members, count, assigned, uninformative, over_limit):
        self.class_off, self.members, self.count = class_off, members, count
        self.assigned, self.uninformative, self.over_limit = assigned, uninformative, over_limit

    def __len__(self):
        return len(self.count)

    def classes(self):
        """[(member tuple, count)] in class order."""
        o = self.class_off
        return [(tuple(int(x) for x in self.members[o[c]:o[c + 1]]), int(self.count[c])) for c in range(len(self))]


class Abundance:
    """What em_abundance reports: ``pi`` float64 [n_haps] (each haplotype's share of the assigned reads), ``n_iter``
    (iterations run), ``converged`` (the last change of pi was <= tol) and ``loglik`` (the sum over classes of
    count * log10 of the class's summed pi)."""

    def __init__(self, pi, n_iter, converged, loglik):
        self.pi, self.n_iter, self.converged, self.loglik = pi, n_iter, converged, loglik


def em_abundance(n_haps, classes, max_iter=10000, tol=1e-12):
    """Each haplotype's share of the reads by EM over read classes (``classes``: a ReadClasses, or a
    (class_off, members, count) triple), in float64 and the fixed operation order of DESIGN.md §4 K7
    (hx_em_abundance; host code, needs no GPU).  -> Abundance."""
    class_off, members, count = _csr(classes)
    pi = np.zeros(max(int(n_haps), 0), dtype=np.float64)
    n_iter, conv, ll = C.c_int32(), C.c_int32(), C.c_double()
    _lib.check(_lib.load().hx_em_abundance(int(n_haps), len(count), class_off.ctypes.data, members.ctypes.data,
                                           count.ctypes.data, int(max_iter), float(tol), pi.ctypes.data,
                                           C.byref(n_iter), C.byref(conv), C.byref(ll)))
    return Abundance(pi, int(n_iter.value), bool(conv.value), float(ll.value))


class Bootstrap:
    """What Hansel.em_bootstrap reports for B replicates over H haplotypes: row 0 is the EM on the classes' counts
    (em_abundance, bit for bit), row b >= 1 the EM on a multinomial resample of the assigned reads (DESIGN.md §4 K8).
    ``pi`` float64 [B+1][H], ``n_iter`` int32 [B+1], ``converged`` bool [B+1], ``loglik`` float64 [B+1], and
    ``count`` int64 [B+1][C] (each row's class counts; row 0 = the input counts) or None."""

    def __init__(self, pi, n_iter, converged, loglik, count=None):
        self.pi, self.n_iter, self.converged, self.loglik, self.count = pi, n_iter, converged, loglik, count


def _csr(classes):
    """A ReadClasses or (class_off, members, count) -> contiguous int64 / int32 / int64 arrays."""
    if isinstance(classes, ReadClasses):
        classes = (classes.class_off, classes.members, classes.count)
    class_off, members, count = classes
    class_off = np.ascontiguousarray(class_off, dtype=np.int64)
    members = np.ascontiguousarray(members, dtype=np.int32)
    count = np.ascontiguousarray(count, dtype=np.int64)
    if len(class_off) != len(count) + 1:
        raise ValueError("class_off must have len(count)+1 entries")
    return class_off, members, count


class PathScores:
    """What Hansel.score_paths reports for H haplotypes over sites 1..N; per-site arrays are [H][N], site s at
    column s-1.  ``weights`` float64 [H][N][8] (the 7 normalised branch weights of Hansel.get_edge_weights_at at the
    site given the haplotype's earlier alleles, 0 for a non-candidate, then the total) or None; ``w_hap`` the weight
    of the haplotype's own allele (0 if it is not a candidate); ``w_second`` the largest weight of the other
    candidates (0 if none); ``best`` uint8 the first-max candidate, the allele the recovery walk would pick there
    (255 where there is no candidate).  Per haplotype: ``loglik`` the sum of log10(w_hap) over the sites with
    w_hap > 0, ``n_unsupported`` the sites with w_hap = 0, ``n_disagree`` the sites where best is not the
    haplotype's allele."""

    NO_CANDIDATE = 255

    def __init__(self, weights, w_hap, w_second, best, loglik, n_unsupported, n_disagree):
        self.weights, self.w_hap, self.w_second, self.best = weights, w_hap, w_second, best
        self.loglik, self.n_unsupported, self.n_disagree = loglik, n_unsupported, n_disagree


class Hansel:
    def __init__(self, symbols, unsymbols, n_snps, band_w=None, device=None, _handle=None,
                 v_site="from", candidates_skip_unsymbols=True):
        symbols = [str(s) for s in symbols]
        unsymbols = [str(s) for s in unsymbols]
        if len(symbols) != 7 or sorted(unsymbols) != sorted([symbols[4], symbols[6]]):
            raise NotImplementedError(
                "the CUDA kernels are specialised to Gretel's alphabet: 7 symbols with "
                "symbols[4] and symbols[6] as the unsymbols (gretel/util.py:83)")
        self.symbols = symbols
        self.unsymbols = unsymbols
        self.symbols_d = {s: s for s in symbols}
        self.symbols_i = {i: s for i, s in enumerate(symbols)}
        self._code = {s: i for i, s in enumerate(symbols)}
        self.n_snps = int(n_snps)
        self.n_slices = 0
        self.n_crumbs = 0
        self.L = 1
        self.v_site = v_site
        self.candidates_skip_unsymbols = candidates_skip_unsymbols
        self.device = _default_device() if device is None else int(device)
        if band_w is None:
            band_w = self.n_snps + 1
            if (self.n_snps + 2) * band_w * 49 * 4 > _DENSE_BAND_LIMIT_BYTES:
                raise ValueError("n_snps=%d needs an explicit band_w (max SNPs per read - 1); "
                                 "a full upper triangle would not be sensible" % self.n_snps)
        self.band_w = max(1, int(band_w))
        self._lib = _lib.load()
        if _handle is None:
            h = C.c_void_p()
            _lib.check(self._lib.hx_create(self.n_snps, self.band_w, self.device, C.byref(h)))
            _handle = h
        self._h = _handle
        self._spill = {}
        self._counts_cache = None

    # ---- construction ----------------------------------------------------------------
    @classmethod
    def init_matrix(cls, symbols, unsymbols, n_snps, band_w=None, device=None, **kw):
        """gretel/util.py:83."""
        return cls(symbols, unsymbols, n_snps, band_w=band_w, device=device, **kw)

    def copy(self):
        """gretel/cmd.py:79 - deep copy on the device, attributes carried over."""
        self.finalize()
        h = C.c_void_p()
        _lib.check(self._lib.hx_copy(self._h, C.byref(h)))
        o = Hansel(self.symbols, self.unsymbols, self.n_snps, band_w=self.band_w, device=self.device,
                   _handle=h, v_site=self.v_site, candidates_skip_unsymbols=self.candidates_skip_unsymbols)
        o.n_slices, o.n_crumbs, o.L = self.n_slices, self.n_crumbs, self.L
        o._spill = dict(self._spill)
        return o

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.hx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- helpers -----------------------------------------------------------------------
    @property
    def flags(self):
        f = 0
        if self.v_site == "to":
            f |= _lib.HX_F_VSITE_TO
        if not self.candidates_skip_unsymbols:
            f |= _lib.HX_F_KEEP_UNSYMBOLS
        return f

    def _touch(self):
        self._counts_cache = None

    def _sym(self, s):
        return self._code[str(s)]

    def encode_path(self, path):
        return np.fromiter((self._code[str(s)] for s in path), dtype=np.uint8, count=len(path))

    def decode_path(self, codes):
        return [self.symbols_d[self.symbols[int(c)]] for c in codes]

    # ---- ingestion ---------------------------------------------------------------------
    def ingest_packed(self, rank, off, codes):
        """Pair-expand packed reads on the GPU (gretel/util.py:226-286).
        Returns cumulative (slices, crumbs, covered_snps, sentinel_increments)."""
        rank = np.ascontiguousarray(rank, dtype=np.int32)
        off = np.ascontiguousarray(off, dtype=np.int64)
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        if len(off) != len(rank) + 1:
            raise ValueError("off must have len(rank)+1 entries")
        totals = np.zeros(4, dtype=np.int64)
        _lib.check(self._lib.hx_ingest_host(self._h, rank.ctypes.data, off.ctypes.data, codes.ctypes.data,
                                            len(rank), totals.ctypes.data))
        self._touch()
        return tuple(int(x) for x in totals)

    def ingest_packed_compact(self, rank, klen, codes4, n_codes):
        """ingest_packed in the compact wire format (see util.compact_packed): uint16 SNP counts and
        nibble-packed codes; offsets and byte codes are rebuilt on the GPU."""
        rank = np.ascontiguousarray(rank, dtype=np.int32)
        klen = np.ascontiguousarray(klen, dtype=np.uint16)
        codes4 = np.ascontiguousarray(codes4, dtype=np.uint8)
        if len(klen) != len(rank) or len(codes4) < (int(n_codes) + 1) // 2:
            raise ValueError("klen/codes4 do not match rank/n_codes")
        totals = np.zeros(4, dtype=np.int64)
        _lib.check(self._lib.hx_ingest_host_compact(self._h, rank.ctypes.data, klen.ctypes.data, codes4.ctypes.data,
                                                    len(rank), int(n_codes), totals.ctypes.data))
        self._touch()
        return tuple(int(x) for x in totals)

    def ingest_packed_dense(self, dense, wait=True):
        """ingest_packed in the dense wire format (util.dense_packed / util.DensePacked).  ``wait=False`` only
        enqueues the chunk (copy on a second stream): call ingest_totals() after the last chunk; the arrays of
        ``dense`` must stay alive and untouched until then."""
        d = dense
        for a in d.arrays():
            if not a.flags["C_CONTIGUOUS"]:
                raise ValueError("dense arrays must be contiguous")
        if len(d.rank_delta) != d.n_reads or len(d.klen) != d.n_reads or len(d.codes2) < (d.n_codes + 3) // 4:
            raise ValueError("dense arrays do not match n_reads/n_codes")
        totals = np.zeros(4, dtype=np.int64)
        if not wait:
            self._dense_keepalive = getattr(self, "_dense_keepalive", []) + [d]
        _lib.check(self._lib.hx_ingest_host_dense(
            self._h, d.rank_delta.ctypes.data, d.esc_idx.ctypes.data, d.esc_delta.ctypes.data, len(d.esc_idx),
            d.klen.ctypes.data, int(d.klen.dtype.itemsize), d.codes2.ctypes.data, d.exc_pos.ctypes.data,
            len(d.exc_pos), d.n_reads, d.n_codes, totals.ctypes.data if wait else None))
        self._touch()
        return tuple(int(x) for x in totals) if wait else None

    def ingest_totals(self):
        totals = np.zeros(4, dtype=np.int64)
        try:
            _lib.check(self._lib.hx_ingest_totals(self._h, totals.ctypes.data))
        finally:
            self._dense_keepalive = []
        return tuple(int(x) for x in totals)

    def set_ingest_kernel(self, which):
        _lib.check(self._lib.hx_set_ingest_kernel(self._h, int(which)))

    def set_ingest_sms(self, n_sms):
        """Leave SMs free for a collective running beside the next batch's pair expansion (0 = use all)."""
        _lib.check(self._lib.hx_set_ingest_sms(self._h, int(n_sms)))

    def set_stream(self, stream_ptr):
        """Order all work of this matrix on an existing CUDA stream (cudaStream_t as int)."""
        _lib.check(self._lib.hx_set_stream(self._h, stream_ptr))

    def counts_buffer(self):
        """(device ptr, n uint32, device ptr, n int64) of the partial counts and totals."""
        a, b = C.c_void_p(), C.c_void_p()
        na, nb = C.c_int64(), C.c_int64()
        _lib.check(self._lib.hx_counts_buffer(self._h, C.byref(a), C.byref(na), C.byref(b), C.byref(nb)))
        return a.value, na.value, b.value, nb.value

    def counts_pack(self, world):
        """(device ptr, n uint32) of the pending counts packed for a cheaper sum all-reduce (hx_counts_pack)."""
        a, na = C.c_void_p(), C.c_int64()
        _lib.check(self._lib.hx_counts_pack(self._h, int(world), C.byref(a), C.byref(na)))
        return a.value, na.value

    def counts_unpack(self):
        """Write the all-reduced packed sums back; False if a lane overflowed (counts untouched)."""
        o = C.c_int32()
        _lib.check(self._lib.hx_counts_unpack(self._h, C.byref(o)))
        self._touch()
        return o.value == 0

    def counts_unpack_async(self, stream=None):
        """Enqueue the write-back of the all-reduced packed sums on ``stream`` (a raw cudaStream_t; default: the
        matrix's own); no synchronisation - see counts_pack_overflowed."""
        _lib.check(self._lib.hx_counts_unpack_async(self._h, C.c_void_p(stream or 0)))
        self._touch()

    def counts_pack_overflowed(self):
        """True if a lane of the last packed exchange overflowed on some rank (its counts were left as partials)."""
        o = C.c_int32()
        _lib.check(self._lib.hx_counts_pack_overflowed(self._h, C.byref(o)))
        return o.value != 0

    def counts_max(self):
        """Largest pending count on this GPU (synchronises)."""
        m = C.c_uint32()
        _lib.check(self._lib.hx_counts_max(self._h, C.byref(m)))
        return int(m.value)

    def ingest_device(self, d_rank_ptr, d_off_ptr, d_codes_ptr, n_reads):
        """Asynchronous ingestion of packed reads already resident on this GPU (raw device pointers)."""
        _lib.check(self._lib.hx_ingest_device(self._h, d_rank_ptr, d_off_ptr, d_codes_ptr, int(n_reads)))
        self._touch()

    def reset_counts(self):
        _lib.check(self._lib.hx_reset_counts(self._h))
        self._touch()

    def probe_expected_rows(self, d_rank_ptr, d_off_ptr, d_codes_ptr, n_reads, d_rows_ptr):
        """Parity probe: add what device-resident reads must leave in every band row into uint64[N+2] at
        ``d_rows_ptr`` (an independent recount of gretel/util.py:254-281; asynchronous on the stream)."""
        _lib.check(self._lib.hx_probe_expected_rows(self._h, d_rank_ptr, d_off_ptr, d_codes_ptr, int(n_reads),
                                                    d_rows_ptr))

    def counts_row_sums(self, d_rows_ptr):
        """Parity probe: row sums of the pending integer counts into uint64[N+2] at ``d_rows_ptr``."""
        _lib.check(self._lib.hx_counts_row_sums(self._h, d_rows_ptr))

    def counts_ipc_export(self, world):
        """Fused exchange, step 1: make the pending counts IPC-shareable; returns the 64-byte handle."""
        buf = C.create_string_buffer(64)
        _lib.check(self._lib.hx_counts_ipc_export(self._h, int(world), buf))
        return bytes(buf.raw)

    def counts_ipc_import(self, handles, my_rank):
        """Fused exchange, step 2: handles = the world handles in rank order (bytes, 64 each)."""
        blob = b"".join(handles)
        _lib.check(self._lib.hx_counts_ipc_import(self._h, blob, len(handles), int(my_rank)))

    def counts_ipc_close(self):
        _lib.check(self._lib.hx_counts_ipc_close(self._h))

    def finalize(self):
        _lib.check(self._lib.hx_finalize_counts(self._h))
        self._touch()

    def sync(self):
        _lib.check(self._lib.hx_sync(self._h))

    @property
    def stream(self):
        s = C.c_void_p()
        _lib.check(self._lib.hx_stream(self._h, C.byref(s)))
        return s.value or 0

    # ---- scalar Hansel surface ---------------------------------------------------------
    def add_observation(self, symbol_from, symbol_to, pos_from, pos_to):
        a, b = self._sym(symbol_from), self._sym(symbol_to)
        rc = self._lib.hx_add_observation(self._h, a, b, int(pos_from), int(pos_to), 1.0)
        if rc == _lib.HX_E_BAND:
            key = (a, b, int(pos_from), int(pos_to))
            self._spill[key] = np.float32(self._spill.get(key, np.float32(0)) + np.float32(1))
        else:
            _lib.check(rc)
        self._touch()

    def get_observation(self, symbol_from, symbol_to, pos_from, pos_to):
        a, b = self._sym(symbol_from), self._sym(symbol_to)
        out = C.c_float()
        rc = self._lib.hx_get_observation(self._h, a, b, int(pos_from), int(pos_to), C.byref(out))
        if rc == _lib.HX_E_BAND:
            return float(self._spill.get((a, b, int(pos_from), int(pos_to)), 0.0))
        _lib.check(rc)
        return float(out.value)

    def reweight_observation(self, symbol_from, symbol_to, pos_from, pos_to, ratio):
        a, b = self._sym(symbol_from), self._sym(symbol_to)
        self.finalize()
        out = C.c_double()
        rc = self._lib.hx_reweight_observation(self._h, a, b, int(pos_from), int(pos_to), float(ratio), C.byref(out))
        if rc == _lib.HX_E_BAND:
            key = (a, b, int(pos_from), int(pos_to))
            old = float(self._spill.get(key, 0.0))
            new = old - float(ratio) * old
            if key in self._spill:
                self._spill[key] = np.float32(new)
            return old - new
        _lib.check(rc)
        self._touch()
        return float(out.value)

    def reweight_matrix(self, ratio):
        self.finalize()
        _lib.check(self._lib.hx_reweight_matrix(self._h, float(ratio)))
        for k in self._spill:
            self._spill[k] = np.float32(float(self._spill[k]) * (1.0 - float(ratio)))
        self._touch()

    def _counts_all(self):
        if self._counts_cache is None:
            self.finalize()
            out = np.zeros((self.n_snps + 1, 8), dtype=np.float64)
            _lib.check(self._lib.hx_counts_all(self._h, out.ctypes.data))
            self._counts_cache = out
        return self._counts_cache

    def get_counts_at(self, at_pos):
        row = self._counts_all()[int(at_pos)]
        d = {self.symbols_d[s]: float(row[i]) for i, s in enumerate(self.symbols) if row[i] > 0}
        d["total"] = float(row[7])
        return d

    def get_marginal_of_at(self, of_symbol, at_pos):
        row = self._counts_all()[int(at_pos)]
        if row[7] == 0:
            return 0.0
        return float(row[self._sym(of_symbol)] / row[7])

    def get_edge_weights_at(self, snp, current_path, debug=False):
        self.finalize()
        path = self.encode_path(current_path[:snp])
        w = np.zeros(7, dtype=np.float64)
        tot, mask = C.c_double(), C.c_int()
        _lib.check(self._lib.hx_edge_weights_at(self._h, int(snp), path.ctypes.data, int(self.L), self.flags,
                                                w.ctypes.data, C.byref(tot), C.byref(mask)))
        out = {self.symbols_d[s]: float(w[i]) for i, s in enumerate(self.symbols) if (mask.value >> i) & 1}
        out["total"] = float(tot.value)
        if debug:
            print(out)
        return out

    # ---- bulk recovery (what gretel_b200.gretel calls) ------------------------------------
    def generate_path_codes(self, original, L=None):
        """-> (codes uint8[N+1], hp_current, hp_original, min_marginal) or (None, hole_site)."""
        self.finalize()
        original.finalize()
        path = np.zeros(self.n_snps + 1, dtype=np.uint8)
        out = np.zeros(3, dtype=np.float64)
        hole = C.c_int32()
        rc = self._lib.hx_generate_path(self._h, original._h, int(self.L if L is None else L), self.flags,
                                        path.ctypes.data, out.ctypes.data, C.byref(hole))
        if rc == _lib.HX_HOLE:
            return None, int(hole.value)
        _lib.check(rc)
        return path, float(out[0]), float(out[1]), float(out[2])

    def reweight_path_codes(self, path_codes, ratio):
        self.finalize()
        path_codes = np.ascontiguousarray(path_codes, dtype=np.uint8)
        if len(path_codes) != self.n_snps + 1:
            raise ValueError("path must have N+1 entries")
        out = C.c_double()
        _lib.check(self._lib.hx_reweight_path(self._h, path_codes.ctypes.data, float(ratio), C.byref(out)))
        self._touch()
        return float(out.value)

    def recover_codes(self, original, max_paths, min_remove=0.01, L=None):
        """Device-resident gretel/cmd.py:148-161 loop -> (paths uint8[n][N+1], stats float64[n][5])."""
        self.finalize()
        original.finalize()
        paths = np.zeros((max_paths, self.n_snps + 1), dtype=np.uint8)
        stats = np.zeros((max_paths, 5), dtype=np.float64)
        n = C.c_int32()
        _lib.check(self._lib.hx_recover(self._h, original._h, int(self.L if L is None else L), self.flags,
                                        int(max_paths), float(min_remove), paths.ctypes.data,
                                        stats.ctypes.data, C.byref(n)))
        self._touch()
        return paths[:n.value], stats[:n.value]

    # ---- read support ------------------------------------------------------------------------
    def assign_reads(self, paths, rank, off, codes, max_mismatch=-1, per_read=False):
        """Assign packed reads to the haplotypes ``paths`` (uint8 [H][N+1], as recover_codes returns them) by the
        fewest mismatches at the read's informative sites; ties split a read equally (hx_assign_reads).  The
        matrix supplies N and the device; its counts are not touched.  -> ReadSupport."""
        paths = np.ascontiguousarray(paths, dtype=np.uint8)
        if paths.ndim != 2 or paths.shape[1] != self.n_snps + 1:
            raise ValueError("paths must be uint8 [n_haps][N+1]")
        rank = np.ascontiguousarray(rank, dtype=np.int32)
        off = np.ascontiguousarray(off, dtype=np.int64)
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        if len(off) != len(rank) + 1:
            raise ValueError("off must have len(rank)+1 entries")
        H, R = paths.shape[0], len(rank)
        unique, shared = np.zeros(H, dtype=np.int64), np.zeros(H, dtype=np.int64)
        share_q32 = np.zeros(H, dtype=np.uint64)
        totals = np.zeros(3, dtype=np.int64)
        per = [np.zeros(R, dtype=np.int32) for _ in range(3)] if per_read else [None] * 3
        _lib.check(self._lib.hx_assign_reads(
            self._h, paths.ctypes.data, H, rank.ctypes.data, off.ctypes.data, codes.ctypes.data, R, int(max_mismatch),
            unique.ctypes.data, shared.ctypes.data, share_q32.ctypes.data, totals.ctypes.data,
            *[a.ctypes.data if a is not None else None for a in per]))
        return ReadSupport(unique, shared, share_q32, int(totals[0]), int(totals[1]), int(totals[2]), *per)

    def read_classes(self, paths, rank, off, codes, max_mismatch=-1):
        """Group the assigned reads into compatibility classes: the reads whose tie sets B (assign_reads) are equal
        form one class (hx_read_classes).  Inputs as for assign_reads; the matrix's counts are not touched.
        -> ReadClasses."""
        paths = np.ascontiguousarray(paths, dtype=np.uint8)
        if paths.ndim != 2 or paths.shape[1] != self.n_snps + 1:
            raise ValueError("paths must be uint8 [n_haps][N+1]")
        rank = np.ascontiguousarray(rank, dtype=np.int32)
        off = np.ascontiguousarray(off, dtype=np.int64)
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        if len(off) != len(rank) + 1:
            raise ValueError("off must have len(rank)+1 entries")
        totals = np.zeros(3, dtype=np.int64)
        n_cls, n_mem = C.c_int64(), C.c_int64()
        _lib.check(self._lib.hx_read_classes(
            self._h, paths.ctypes.data, paths.shape[0], rank.ctypes.data, off.ctypes.data, codes.ctypes.data,
            len(rank), int(max_mismatch), totals.ctypes.data, C.byref(n_cls), C.byref(n_mem)))
        class_off = np.zeros(n_cls.value + 1, dtype=np.int64)
        members = np.zeros(n_mem.value, dtype=np.int32)
        count = np.zeros(n_cls.value, dtype=np.int64)
        _lib.check(self._lib.hx_read_classes_get(self._h, class_off.ctypes.data, members.ctypes.data,
                                                 count.ctypes.data))
        return ReadClasses(class_off, members, count, int(totals[0]), int(totals[1]), int(totals[2]))

    def em_bootstrap(self, n_haps, classes, n_boot, seed=0, max_iter=10000, tol=1e-12, counts=False):
        """Bootstrap of the abundance EM on the GPU (hx_em_bootstrap): row 0 is em_abundance on ``classes`` (a
        ReadClasses or a (class_off, members, count) triple), row b = 1..n_boot the same EM on the counts of a
        resample of the assigned reads with replacement, drawn by Philox4x32-10 keyed by ``seed`` (uint64).  Every row
        depends only on (classes, seed, b).  The matrix supplies the device; its counts are not touched.
        -> Bootstrap (``count`` with counts=True)."""
        class_off, members, count = _csr(classes)
        H, R, Cn = max(int(n_haps), 0), max(int(n_boot), 0) + 1, len(count)
        pi = np.zeros((R, H), dtype=np.float64)
        n_iter, conv = np.zeros(R, dtype=np.int32), np.zeros(R, dtype=np.int32)
        ll = np.zeros(R, dtype=np.float64)
        cnt = np.zeros((R, Cn), dtype=np.int64) if counts else None
        _lib.check(self._lib.hx_em_bootstrap(
            self._h, int(n_haps), Cn, class_off.ctypes.data, members.ctypes.data, count.ctypes.data, int(n_boot),
            int(seed) & 0xFFFFFFFFFFFFFFFF, int(max_iter), float(tol), pi.ctypes.data, n_iter.ctypes.data,
            conv.ctypes.data, ll.ctypes.data, cnt.ctypes.data if counts else None))
        return Bootstrap(pi, n_iter, conv.astype(bool), ll, cnt)

    # ---- path scores --------------------------------------------------------------------------
    def score_paths(self, paths, L=None, weights=False):
        """Score the haplotypes ``paths`` (uint8 [H][N+1] as recover_codes returns them: '_' at site 0, codes 0..6)
        against this matrix: at every site the branch weights of get_edge_weights_at given the haplotype's earlier
        alleles, with ``L`` (default: the matrix's L) and the matrix's flags, as recovery uses them (hx_score_paths).
        The matrix is not changed.  -> PathScores."""
        self.finalize()
        paths = np.ascontiguousarray(paths, dtype=np.uint8)
        if paths.ndim != 2 or paths.shape[1] != self.n_snps + 1:
            raise ValueError("paths must be uint8 [n_haps][N+1]")
        H, N = paths.shape[0], self.n_snps
        w = np.zeros((H, N, 8), dtype=np.float64) if weights else None
        w_hap, w_second = np.zeros((H, N), dtype=np.float64), np.zeros((H, N), dtype=np.float64)
        best = np.zeros((H, N), dtype=np.uint8)
        loglik = np.zeros(H, dtype=np.float64)
        n_unsup, n_dis = np.zeros(H, dtype=np.int32), np.zeros(H, dtype=np.int32)
        _lib.check(self._lib.hx_score_paths(
            self._h, paths.ctypes.data, H, int(self.L if L is None else L), self.flags,
            w.ctypes.data if w is not None else None, w_hap.ctypes.data, w_second.ctypes.data, best.ctypes.data,
            loglik.ctypes.data, n_unsup.ctypes.data, n_dis.ctypes.data))
        return PathScores(w, w_hap, w_second, best, loglik, n_unsup, n_dis)

    # ---- bulk I/O ----------------------------------------------------------------------------
    def band(self):
        """float32 [N+2][W][7][7]; cell (pi,pj) at [pj][pj-pi-1]."""
        self.finalize()
        out = np.zeros((self.n_snps + 2, self.band_w, 7, 7), dtype=np.float32)
        _lib.check(self._lib.hx_band_to_host(self._h, out.ctypes.data))
        return out

    def load_band(self, band):
        self.finalize()
        band = np.ascontiguousarray(band, dtype=np.float32)
        if band.shape != (self.n_snps + 2, self.band_w, 7, 7):
            raise ValueError("band shape mismatch")
        _lib.check(self._lib.hx_band_from_host(self._h, band.ctypes.data))
        self._touch()

    def to_dense(self):
        """float32 (7,7,N+2,N+2) like the reference's ndarray (small N only)."""
        self.finalize()
        P = self.n_snps + 2
        out = np.zeros((7, 7, P, P), dtype=np.float32)
        _lib.check(self._lib.hx_to_dense(self._h, out.ctypes.data))
        for (a, b, i, j), v in self._spill.items():
            out[a, b, i, j] = v
        return out

    def save_hansel_dump(self, path):
        """gretel/cmd.py:82.  Format (ours; upstream's is defined in un-vendored hansel):
        .npz with the float32 band and the attributes."""
        np.savez_compressed(path, band=self.band(), n_snps=self.n_snps, band_w=self.band_w, L=self.L,
                            n_slices=self.n_slices, n_crumbs=self.n_crumbs, symbols=np.array(self.symbols),
                            unsymbols=np.array(self.unsymbols))

    @classmethod
    def load_hansel_dump(cls, path, device=None):
        z = np.load(path if str(path).endswith(".npz") else str(path) + ".npz")
        h = cls([str(s) for s in z["symbols"]], [str(s) for s in z["unsymbols"]], int(z["n_snps"]),
                band_w=int(z["band_w"]), device=device)
        h.load_band(z["band"])
        h.L, h.n_slices, h.n_crumbs = int(z["L"]), int(z["n_slices"]), int(z["n_crumbs"])
        return h

    def kernel_ms(self, which):
        ms = C.c_float()
        _lib.check(self._lib.hx_last_kernel_ms(self._h, {"ingest": 0, "walk": 1, "reweight": 2, "assign": 3,
                                                                "score": 4, "classes": 5, "resample": 6,
                                                                "bootstrap_em": 7}[which],
                                               C.byref(ms)))
        return float(ms.value)

    def launch_count(self):
        n = C.c_int64()
        _lib.check(self._lib.hx_launch_count(self._h, C.byref(n)))
        return int(n.value)
