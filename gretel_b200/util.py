"""Ingestion entry points with the reference's names and argument meaning.

``load_from_bam`` / ``process_vcf`` / ``get_ref_len_from_bam`` mirror
gretel/util.py:33, :354, :10 of the reference.  BAM/VCF parsing stays on the CPU
(north_star) and produces the packed ``(rank, off, codes)`` arrays; the pair expansion
(util.py:226-286) runs in the CUDA ingestion kernel.
"""
from __future__ import annotations

import sys
from math import ceil

import numpy as np

from . import bamio
from .bamio import get_ref_len_from_bam, process_vcf  # noqa: F401  (re-exported, same names as the reference)
from .hansel import Hansel, REF_SYMBOLS, REF_UNSYMBOLS


def band_width_for(off, floor=1):
    """Smallest band that holds every pair of every read: max SNPs on a read - 1."""
    off = np.asarray(off)
    if len(off) < 2:
        return max(1, floor)
    return max(int(np.diff(off).max()) - 1, floor, 1)


def compact_packed(off, codes):
    """(off int64[R+1], codes uint8) -> (klen uint16[R], codes4 uint8[ceil(n/2)], n_codes): the compact
    wire format of Hansel.ingest_packed_compact (two allele codes per byte, low nibble first)."""
    off = np.asarray(off, dtype=np.int64)
    k = np.diff(off)
    if len(k) and k.max() > 65535:
        raise ValueError("a read covers more than 65535 SNPs")
    c = np.ascontiguousarray(codes[off[0]:off[-1]] if len(off) else codes, dtype=np.uint8)
    n = len(c)
    if n & 1:
        c = np.concatenate([c, np.zeros(1, np.uint8)])
    codes4 = (c[0::2] | (c[1::2] << 4)).astype(np.uint8)
    return k.astype(np.uint16), codes4, n


class DensePacked:
    """Rank-sorted packed reads in the dense wire format of hx_ingest_host_dense (include/hanselx.h): uint8 rank
    deltas (255 = listed in esc_idx/esc_delta), uint8|uint16 SNP counts, 2-bit alleles with the N/-/_ positions
    listed in exc_pos.  ``chunks(n)`` splits at read boundaries for the overlapped (asynchronous) ingestion."""
    __slots__ = ("rank_delta", "esc_idx", "esc_delta", "klen", "codes2", "exc_pos", "n_reads", "n_codes", "blob")

    def __init__(self, rank_delta, esc_idx, esc_delta, klen, codes2, exc_pos, n_reads, n_codes):
        self.rank_delta, self.esc_idx, self.esc_delta = rank_delta, esc_idx, esc_delta
        self.klen, self.codes2, self.exc_pos = klen, codes2, exc_pos
        self.n_reads, self.n_codes = int(n_reads), int(n_codes)
        self.blob = None            # the single host buffer the arrays are views of (dense_packed), if any

    def rebased(self, blob):
        """The same chunk as views of ``blob`` (a copy of self.blob, e.g. in pinned memory)."""
        base = self.blob.ctypes.data
        def view(a):
            o = a.ctypes.data - base
            return blob[o:o + a.nbytes].view(a.dtype)
        out = DensePacked(*[view(a) for a in self.arrays()], self.n_reads, self.n_codes)
        out.blob = blob
        return out

    @property
    def nbytes(self):
        return sum(int(a.nbytes) for a in (self.rank_delta, self.esc_idx, self.esc_delta, self.klen, self.codes2,
                                           self.exc_pos))

    def arrays(self):
        return (self.rank_delta, self.esc_idx, self.esc_delta, self.klen, self.codes2, self.exc_pos)


def dense_packed_native(rank, off, codes, n_threads=8):
    """dense_packed by the C++ encoder of libhanselx.so (hx_dense_encode); byte-identical output."""
    import ctypes as C

    from . import _lib
    lib = _lib.load()
    rank = np.ascontiguousarray(rank, dtype=np.int32)
    off = np.ascontiguousarray(off, dtype=np.int64)
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    if len(off) != len(rank) + 1:
        raise ValueError("off must have len(rank)+1 entries")
    out = _lib.HxDense()
    rc = lib.hx_dense_encode(rank.ctypes.data, off.ctypes.data, codes.ctypes.data, len(rank), int(n_threads), C.byref(out))
    if rc == _lib.HX_E_ARG:
        raise ValueError(lib.hx_last_error().decode())
    _lib.check(rc)
    try:
        blob = np.ctypeslib.as_array(out.blob, shape=(int(out.blob_bytes),)).copy()
        R, n, kb = int(out.n_reads), int(out.n_codes), int(out.klen_bytes)
        d = DensePacked(blob[0:R],
                        blob[out.o_esc_idx:out.o_esc_idx + 8 * out.n_esc].view(np.int64),
                        blob[out.o_esc_delta:out.o_esc_delta + 4 * out.n_esc].view(np.int32),
                        blob[out.o_klen:out.o_klen + R * kb].view(np.uint8 if kb == 1 else np.uint16),
                        blob[out.o_codes2:out.o_codes2 + (n + 3) // 4],
                        blob[out.o_exc:out.o_exc + 4 * out.n_exc].view(np.uint32), R, n)
        d.blob = blob
    finally:
        lib.hx_dense_free(C.byref(out))
    return d


def dense_packed(rank, off, codes):
    """(rank int32[R] non-decreasing, off int64[R+1], codes uint8) -> DensePacked (numpy encoder)."""
    rank = np.asarray(rank, dtype=np.int64)
    off = np.asarray(off, dtype=np.int64)
    k = np.diff(off)
    d = np.diff(rank, prepend=0)
    if len(d) and d.min() < 0:
        raise ValueError("the dense wire format needs reads sorted by rank")
    if len(k) and k.max() > 65535:
        raise ValueError("a read covers more than 65535 SNPs")
    esc_idx = np.nonzero(d >= 255)[0].astype(np.int64)
    c = np.ascontiguousarray(codes[off[0]:off[-1]] if len(off) else codes, dtype=np.uint8)
    n = len(c)
    if n >= 1 << 32:
        raise ValueError("more than 2^32 alleles in one call: split the reads into chunks")
    if n and c.max() > 6:
        raise ValueError("allele code > 6")
    exc = np.nonzero(c >= 4)[0].astype(np.uint32)
    f = np.where(c >= 4, c - 4, c).astype(np.uint8)
    if n & 3:
        f = np.concatenate([f, np.zeros(4 - (n & 3), np.uint8)])
    # one host buffer laid out like the device staging set (16-byte aligned sections, wire.cu), so that the
    # library ships it with a single copy
    R, kb = len(k), (1 if (len(k) == 0 or k.max() < 256) else 2)
    al = lambda x: (int(x) + 15) & ~15
    n_words = (n + 15) // 16
    o_kl = al(R)
    o_c2 = o_kl + al(R * kb)
    o_ex = o_c2 + al(n_words * 4)
    o_ei = o_ex + al(len(exc) * 4)
    o_ed = o_ei + al(len(esc_idx) * 8)
    blob = np.zeros(o_ed + al(len(esc_idx) * 4) + 16, dtype=np.uint8)
    rank_delta = blob[0:R]
    rank_delta[:] = np.minimum(d, 255)
    klen = blob[o_kl:o_kl + R * kb].view(np.uint8 if kb == 1 else np.uint16)
    klen[:] = k
    codes2 = blob[o_c2:o_c2 + (n + 3) // 4]
    codes2[:] = f[0::4] | (f[1::4] << 2) | (f[2::4] << 4) | (f[3::4] << 6)
    exc_pos = blob[o_ex:o_ex + 4 * len(exc)].view(np.uint32)
    exc_pos[:] = exc
    ei = blob[o_ei:o_ei + 8 * len(esc_idx)].view(np.int64)
    ei[:] = esc_idx
    ed = blob[o_ed:o_ed + 4 * len(esc_idx)].view(np.int32)
    ed[:] = d[esc_idx]
    out = DensePacked(rank_delta, ei, ed, klen, codes2, exc_pos, R, n)
    out.blob = blob
    return out


def dense_chunks(rank, off, codes, n_chunks, weights=None, native=False, n_threads=8):
    """Split rank-sorted packed reads into DensePacked pieces at read boundaries: ``n_chunks`` pieces of about
    equal allele count, or pieces proportional to ``weights`` (a shorter last piece shortens the part of the
    pipeline that cannot overlap a copy)."""
    off = np.asarray(off, dtype=np.int64)
    R = len(off) - 1
    if weights is None:
        n_chunks = max(1, min(int(n_chunks), max(R, 1)))
        weights = [1.0] * n_chunks
    w = np.cumsum(np.asarray(weights, dtype=np.float64))
    targets = off[0] + ((off[-1] - off[0]) * (w[:-1] / w[-1])).astype(np.int64)
    cuts = [0] + [int(x) for x in np.searchsorted(off, targets, side="left")] + [R]
    enc = (lambda r, o, c: dense_packed_native(r, o, c, n_threads=n_threads)) if native else dense_packed
    out = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        if b > a:
            out.append(enc(rank[a:b], off[a:b + 1], codes))
    return out


DENSE_MIN_READS = 200_000      # below this the host->device copy is not what bounds ingestion
DENSE_CHUNK_CODES = 40_000_000


def load_from_packed(rank, off, codes, n_snps, band_w=None, device=None, hansel=None, finalize=True,
                     quiet=True, wire="auto", n_threads=8):
    """Packed reads -> Hansel (util.py:83 + 226-286 + 329-333).

    With ``finalize=False`` the integer counts stay pending so that partial matrices of
    several GPUs can be summed first (see gretel_b200.dist).  ``wire``: "auto" hands the packed arrays to
    hx_ingest_host (large inputs go in a few chunks, each expanded while the next is copied; with
    HX_HOST_PIPELINE=dense the host threads re-encode them into the dense wire format first, which pays on hosts
    with many cores); "dense" does that re-encoding chunk by chunk from Python (hx_dense_encode +
    hx_ingest_host_dense)."""
    if hansel is None:
        if band_w is None:
            band_w = band_width_for(off)
        hansel = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, n_snps, band_w=band_w, device=device)
    rank = np.asarray(rank)
    if wire == "dense":
        off = np.asarray(off, dtype=np.int64)
        n_chunks = max(2, int((off[-1] - off[0]) // DENSE_CHUNK_CODES) + 1) if len(rank) > 1 else 1
        targets = off[0] + (off[-1] - off[0]) * np.arange(1, n_chunks) // n_chunks
        cuts = [0] + [int(x) for x in np.searchsorted(off, targets, side="left")] + [len(rank)]
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b > a:
                hansel.ingest_packed_dense(dense_packed_native(rank[a:b], off[a:b + 1], codes, n_threads=n_threads),
                                           wait=False)
        slices, crumbs, covered, _sent = hansel.ingest_totals()
    else:
        slices, crumbs, covered, _sent = hansel.ingest_packed(rank, off, codes)
    if finalize:
        hansel.finalize()
        set_totals(hansel, slices, crumbs, covered, quiet=quiet)
    return hansel


def set_totals(hansel, slices, crumbs, covered, quiet=True):
    """util.py:329-333."""
    hansel.n_slices = int(slices)
    hansel.n_crumbs = int(crumbs)
    if not quiet:
        sys.stderr.write("[NOTE] Loaded %d breadcrumbs from %d bread slices.\n" % (hansel.n_crumbs, hansel.n_slices))
    hansel.L = int(ceil(float(covered) / slices))        # ZeroDivisionError like the reference if no read has >=2 SNPs
    if not quiet:
        sys.stderr.write("[NOTE] Setting Gretel.L to %d\n" % hansel.L)
    return hansel


def load_from_bam(bam_path, target_contig, start_pos, end_pos, vcf_handler, use_end_sentinels=False,
                  n_threads=1, debug_reads=False, debug_pos=False, stepper="samtools", device=None,
                  band_w=None, max_depth=bamio.PYSAM_MAX_DEPTH, stages=None, reads=None):
    """gretel/util.py:33.  Same signature and return value; ``n_threads`` is accepted for
    compatibility (the reference's window sharding is replaced by one GPU kernel and the
    result is independent of it, cf. tests/test_test.py:35).  ``use_end_sentinels`` is an
    experimental dead branch upstream (never passed, cmd.py:78) and is rejected here.  ``max_depth``: the
    reference reads the BAM through pysam's pileup, whose buffer drops reads beyond 8000 per position
    (bamio._DepthCap); the default reproduces that, ``max_depth=0`` keeps every read.  ``stages``: dict that
    receives per-stage seconds of the packer and of the GPU ingestion.  ``reads``: dict that receives the packed
    reads ``rank``, ``off`` and ``codes`` (for Hansel.assign_reads)."""
    if use_end_sentinels:
        raise NotImplementedError("use_end_sentinels is never enabled by the reference (cmd.py:28,78)")
    # n_threads (the reference's number of BAM iterators, cmd.py:31) drives the native packer's threads
    import time
    t0 = time.perf_counter()
    rank, off, codes = bamio.pack_bam_native(bam_path, target_contig, start_pos, end_pos, vcf_handler,
                                             stepper=stepper, n_threads=n_threads, max_depth=max_depth, stages=stages)
    t1 = time.perf_counter()
    if band_w is None:
        # hold every ingested pair; at least N+1 for tiny regions so that the scalar API
        # (add/get_observation on arbitrary i<j) is band-resident like the reference's dense array
        band_w = band_width_for(off)
        if vcf_handler["N"] <= 256:
            band_w = max(band_w, vcf_handler["N"] + 1)
    h = load_from_packed(rank, off, codes, vcf_handler["N"], band_w=band_w, device=device, quiet=False,
                         n_threads=max(1, n_threads))
    if reads is not None:
        reads.update(rank=rank, off=off, codes=codes)
    if stages is not None:
        stages["pack_total"] = t1 - t0
        stages["gpu_ingest"] = time.perf_counter() - t1
        stages["reads"] = int(len(rank))
    return h
