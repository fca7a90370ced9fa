"""Synthetic packed-read generators for BASELINE.json configs 2-5 (SURVEY.md section 8d).

All draws come from ``numpy.random.Generator(PCG64(seed))`` with
``seed = 20260000 + config#`` (+ rank for per-GPU shards), so the oracle, the tests
and the bench see identical inputs.  Output is the packed format the CUDA path
consumes directly: ``rank int32[R]`` (0-based index of the first SNP on the read),
``off int64[R+1]``, ``codes uint8[sum k]`` with codes A0 C1 G2 T3 N4 -5 _6
(order fixed by gretel/util.py:83); reads are sorted by start (=> by rank) and reads
covering fewer than two SNPs are dropped (util.py:230).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

ABUNDANCES = np.array([0.40, 0.25, 0.15, 0.12, 0.08])


@dataclass(frozen=True)
class Workload:
    name: str
    config: int          # BASELINE.json configs[] index
    genome_len: int      # G
    n_snps: int          # N
    n_reads: int         # R (before dropping reads with <2 SNPs)
    read_len: int        # mean length for long reads
    eps: float           # substitution rate per covered SNP
    delta: float         # deletion rate per covered SNP
    long_reads: bool = False


WORKLOADS = {
    # C2: synthetic HIV-1-like 9.7 kb contig, 5 strains, ~1k SNPs, 200k x 250 bp reads
    "hiv": Workload("hiv", 1, 9_700, 1_000, 200_000, 250, 0.005, 0.001),
    # C3: synthetic metagenomic gene region, 10k SNPs, 10M x 150 bp reads
    "metagenome": Workload("metagenome", 2, 100_000, 10_000, 10_000_000, 150, 0.005, 0.001),
    # between the configs: 1M x 800 bp reads, ~80 SNPs/read (wider than the bit-sliced / tensor-core kernels take,
    # far narrower than ONT: the regime VERDICT r1 asked to measure; not a BASELINE config)
    "mid": Workload("mid", 2, 100_000, 10_000, 1_000_000, 800, 0.005, 0.001),
    # C4: 100k x 10 kb ONT-like reads, ~300 SNPs/read
    "ont": Workload("ont", 3, 333_000, 10_000, 100_000, 10_000, 0.05, 0.02, long_reads=True),
}


def scaled(w: Workload, n_reads: int) -> Workload:
    return Workload(w.name, w.config, w.genome_len, w.n_snps, int(n_reads), w.read_len,
                    w.eps, w.delta, w.long_reads)


def make_strains(rng, n_snps, n_strains=5):
    """Per site 2-3 distinct alleles from ACGT, assigned so that >=2 strains differ."""
    n_alleles = rng.integers(2, 4, size=n_snps)                   # 2 or 3
    perm = np.argsort(rng.random((n_snps, 4)), axis=1)            # random allele order per site
    assign = rng.integers(0, 3, size=(n_strains, n_snps)) % n_alleles[None, :]
    # force strains 0 and 1 onto different alleles so every site is polymorphic
    assign[0, :] = 0
    assign[1, :] = 1
    strains = np.take_along_axis(perm.T, assign, axis=0)          # [S][N] codes 0..3
    return np.ascontiguousarray(strains, dtype=np.uint8)


def make_sites(rng, genome_len, n_snps):
    return np.sort(rng.choice(genome_len, size=n_snps, replace=False) + 1).astype(np.int64)


def generate(w: Workload, seed=None, shard=0, chunk=2_000_000):
    """Return dict(rank, off, codes, n_snps, sites, strains, max_k, n_pairs, strain_of); strain_of[i] is the
    strain read i was drawn from."""
    if seed is None:
        seed = 20260000 + w.config + 1
    # strains/sites depend on the workload seed only; reads also on the shard so that
    # every GPU of a weak-scaling run ingests a different slice of the same metagenome.
    rng_g = np.random.Generator(np.random.PCG64(seed))
    sites = make_sites(rng_g, w.genome_len, w.n_snps)
    strains = make_strains(rng_g, w.n_snps)
    rng = np.random.Generator(np.random.PCG64([seed, 7919 + shard]))
    R, G = w.n_reads, w.genome_len
    if w.long_reads:
        sigma = 0.3
        mu = np.log(w.read_len) - 0.5 * sigma * sigma
        lens = np.clip(rng.lognormal(mu, sigma, size=R), 2_000, 30_000).astype(np.int64)
    else:
        lens = np.full(R, w.read_len, dtype=np.int64)
    start = rng.integers(1 - w.read_len + 1, G + 1, size=R)
    order = np.argsort(start, kind="stable")
    start = start[order]
    lens = lens[order]
    s = np.maximum(start, 1)
    e = np.minimum(start + lens - 1, G)
    rank = np.searchsorted(sites, s, side="left")
    hi = np.searchsorted(sites, e, side="right")
    k = hi - rank
    keep = k >= 2
    rank, k = rank[keep].astype(np.int64), k[keep].astype(np.int64)
    strain_of = rng.choice(len(ABUNDANCES), size=R, p=ABUNDANCES)[keep].astype(np.int64)
    off = np.zeros(len(k) + 1, dtype=np.int64)
    np.cumsum(k, out=off[1:])
    total = int(off[-1])
    codes = np.empty(total, dtype=np.uint8)
    flat_strains = strains.reshape(-1)
    N = w.n_snps
    # chunk the flat expansion to bound temporaries (150 M codes for C3)
    r0 = 0
    nreads = len(k)
    while r0 < nreads:
        r1 = min(nreads, r0 + chunk)
        kk = k[r0:r1]
        n = int(off[r1] - off[r0])
        rep = np.repeat(np.arange(r1 - r0), kk)
        t = np.arange(n, dtype=np.int64) - np.repeat(off[r0:r1] - off[r0], kk)
        site = rank[r0:r1][rep] + t
        c = flat_strains[strain_of[r0:r1][rep] * N + site]
        u = rng.random(n, dtype=np.float32)
        sub = u < w.eps
        if sub.any():
            shift = rng.integers(1, 4, size=int(sub.sum())).astype(np.uint8)
            c[sub] = (c[sub] + shift) % 4
        c[(u >= w.eps) & (u < w.eps + w.delta)] = 5                # '-'
        c[(u >= w.eps + w.delta) & (u < w.eps + w.delta + 0.001)] = 4   # 'N'
        codes[off[r0]:off[r1]] = c
        r0 = r1
    return {
        "rank": rank.astype(np.int32), "off": off, "codes": codes, "n_snps": N,
        "sites": sites, "strains": strains, "max_k": int(k.max()) if len(k) else 0,
        "n_pairs": int((k * (k - 1) // 2).sum()), "strain_of": strain_of,
    }


def random_packed(rng, n_snps, n_reads, max_k, p_special=0.1, sort=True):
    """Small adversarial packed reads for parity tests: any code 0..6, k in [0, max_k]."""
    ks = rng.integers(0, max_k + 1, size=n_reads)
    ks = np.minimum(ks, n_snps)
    ranks = np.array([rng.integers(0, n_snps - k + 1) for k in ks], dtype=np.int64)
    if sort:
        o = np.argsort(ranks, kind="stable")
        ranks, ks = ranks[o], ks[o]
    off = np.zeros(n_reads + 1, dtype=np.int64)
    np.cumsum(ks, out=off[1:])
    codes = rng.integers(0, 4, size=int(off[-1])).astype(np.uint8)
    special = rng.random(len(codes)) < p_special
    codes[special] = rng.integers(4, 7, size=int(special.sum())).astype(np.uint8)
    return ranks.astype(np.int32), off, codes


def write_bam(path, d, w, contig="ctg", threads=8, level=1):
    """Write the reads of a ``generate()`` result as a coordinate-sorted BAM (fixed-length 150M reads; vectorised,
    so a million reads take seconds).  The reference base is 'A' everywhere; a read carries its packed alleles at
    the SNP sites it covers ('-' cannot be expressed in a fixed-length all-match record and is written as 'N').
    Returns ``(vcf_handler, keep)``: the dict process_vcf() would build for the region [1, genome_len] and the
    mask of the reads that were written (reads clipped by the genome's ends are not)."""
    import struct
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    if w.long_reads:
        raise ValueError("write_bam: short-read workloads only")
    sites, rank, off, codes = d["sites"], d["rank"].astype(np.int64), d["off"], d["codes"]
    R, L, G = len(rank), int(w.read_len), int(w.genome_len)
    k = np.diff(off)
    # a read starts somewhere in (sites[rank-1], sites[rank]] and must cover exactly its k SNPs
    last_site = sites[rank + k - 1]
    nxt = np.where(rank + k < len(sites), sites[np.minimum(rank + k, len(sites) - 1)], G + L + 1)
    lo = np.maximum(np.where(rank > 0, sites[np.maximum(rank - 1, 0)] + 1, 1), np.maximum(last_site - L + 1, 1))
    hi = np.minimum(sites[rank], nxt - L)
    # reads clipped by the ends of the genome cannot be full-length all-match records: they are left out
    keep = (lo <= hi) & (lo + L - 1 <= G)
    rank, k, start = rank[keep], k[keep], lo[keep]            # 1-based start
    sel = np.repeat(keep, np.diff(off))
    codes = codes[sel]
    off = np.concatenate([[0], np.cumsum(k)])
    R = len(rank)
    order = np.argsort(start, kind="stable")
    name_len = 10                                             # 9 characters + NUL
    rec = 4 + 32 + name_len + 4 + (L + 1) // 2 + L
    buf = np.zeros((R, rec), dtype=np.uint8)
    def put32(col, vals):
        buf[:, col:col + 4] = np.ascontiguousarray(vals, dtype="<i4").view(np.uint8).reshape(-1, 4)
    put32(0, np.full(R, rec - 4))
    put32(4, np.zeros(R))                                     # refID
    put32(8, start - 1)                                       # pos (0-based)
    buf[:, 12] = name_len
    buf[:, 13] = 42                                           # mapq
    buf[:, 14:16] = np.array([4680 & 0xff, 4680 >> 8], np.uint8)
    buf[:, 16:18] = np.array([1, 0], np.uint8)                # n_cigar_op
    buf[:, 18:20] = 0                                         # flag
    put32(20, np.full(R, L))
    put32(24, np.full(R, -1)); put32(28, np.full(R, -1)); put32(32, np.zeros(R))
    ids = np.arange(R)
    name = np.zeros((R, name_len), np.uint8)
    name[:, 0] = ord("r")
    for j in range(8):
        name[:, 8 - j] = ord("0") + (ids // 10 ** j) % 10
    buf[:, 36:36 + name_len] = name
    buf[:, 36 + name_len:40 + name_len] = np.array([(L << 4) & 0xff, (L << 4) >> 8 & 0xff, 0, 0], np.uint8)
    # bases: 'A' (1) everywhere, the packed alleles at the covered SNP sites
    nt16 = np.array([1, 2, 4, 8, 15, 15, 15], np.uint8)       # A C G T N -(as N) _
    bases = np.full((R, L + (L & 1)), 1, dtype=np.uint8)
    rep = np.repeat(np.arange(R), k)
    t = np.arange(len(codes)) - np.repeat(off[:-1], k)
    col = sites[np.repeat(rank, k) + t] - start[rep]
    bases[rep, col] = nt16[codes]
    if L & 1:
        bases[:, L] = 0
    seq_at = 40 + name_len
    buf[:, seq_at:seq_at + (L + 1) // 2] = (bases[:, 0::2] << 4) | bases[:, 1::2]
    # base qualities: random (they dominate the size of a real BAM and the cost of inflating it)
    buf[:, seq_at + (L + 1) // 2:] = np.random.default_rng(7).integers(2, 41, size=(R, L), dtype=np.uint8)
    text = "@HD\tVN:1.0\tSO:coordinate\n@SQ\tSN:%s\tLN:%d\n" % (contig, G)
    head = (b"BAM\x01" + struct.pack("<i", len(text)) + text.encode() + struct.pack("<i", 1)
            + struct.pack("<i", len(contig) + 1) + contig.encode() + b"\x00" + struct.pack("<i", G))
    body = buf[order].tobytes()
    def bgzf(chunk):
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        comp = co.compress(chunk) + co.flush()
        return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(comp) + 25)
                + comp + struct.pack("<II", zlib.crc32(chunk) & 0xffffffff, len(chunk)))
    # as htslib writes it: the header in a block of its own, and a block ends rather than cut a record
    blk = (65280 // rec) * rec
    chunks = [head] + [body[i:i + blk] for i in range(0, len(body), blk)]
    with ThreadPoolExecutor(max_workers=max(1, threads)) as ex, open(path, "wb") as fh:
        for b in ex.map(bgzf, chunks, chunksize=64):
            fh.write(b)
        fh.write(bgzf(b""))
    region = np.zeros(G + 1, dtype=int)
    region[sites] = 1
    vh = {"N": len(sites), "snp_fwd": {int(p): i for i, p in enumerate(sites)},
          "snp_rev": {i: int(p) for i, p in enumerate(sites)}, "region": region}
    return vh, keep
