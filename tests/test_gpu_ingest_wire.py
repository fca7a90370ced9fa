"""Host-to-device ingestion where its wire formats and pipelines change regime, against the C oracle.

Between the caller's (rank, off, codes) arrays and the pair-expansion kernels sit the dense wire format (uint8 rank
deltas with an escape list, uint8 / uint16 SNP counts, 2-bit alleles with an exception list), its three decode
kernels (k_dense_partials, k_dense_spine, k_dense_apply), the host pipelines of hx_ingest_host (slim: allele bytes as
they are; dense: re-encoded), their pinned slots and staging sets, and the compact path's scan.  Each case here
reaches a regime the small inputs of test_gpu_ingest never do: a spine longer than one step of 1024 blocks (4,194,304
reads), escapes and rank runs on the 16-read and 4096-read decode granules, more than six pipeline chunks, buffers
that grow while other chunks are in flight, the uint16 SNP counts a band of W + 1 >= 256 selects, slices with
absolute offsets.  Every result is compared with the C oracle: the float32 band bit for bit and all four totals.
Bad reads must be refused with the same status at every input size and under every HX_HOST_PIPELINE."""
import numpy as np
import pytest

from tests.test_gpu_ingest_launch import _add, _assert_band, _case, _totals

pytestmark = pytest.mark.gpu

SPINE_STEP = 1024 * 4096            # reads (+ the entry off[n]) one k_dense_spine step covers
CHUNK_CODES = 32 << 20              # alleles per chunk of hx_ingest_host's pipeline (wire.cu)
PIPELINE_MIN_READS = 200_000        # hx_ingest_host pipelines inputs of this many reads and more


# ---- inputs ----------------------------------------------------------------------------------------------------------

def _codes(rng, n, p_special):
    """n random allele codes, a fraction p_special of them N / - / _ (codes 4..6); one byte of randomness each."""
    x = rng.integers(0, 256, size=n, dtype=np.uint8)
    codes = x & 3
    sp = x < int(round(p_special * 256))
    codes[sp] = 4 + x[sp] % 3
    return codes


def _reads(k, d, rng, p_special=0.05, pad=0, N=None):
    """Rank-sorted packed reads of k[i] SNPs at rank[i] = d[0] + ... + d[i]; N = the last site a read reaches + pad,
    unless given."""
    rank = np.cumsum(d)
    reach = int((rank + k).max())
    assert N is None or reach <= N
    N = reach + pad if N is None else N
    off = np.zeros(len(k) + 1, np.int64)
    np.cumsum(k, out=off[1:])
    return rank.astype(np.int32), off, _codes(rng, int(off[-1]), p_special), N


def _steps(rng, d, n_steps):
    """A rank step of 1 before about n_steps random reads that have none yet (rank runs of random length)."""
    at = rng.integers(1, len(d), size=n_steps)
    d[at] = np.maximum(d[at], 1)


def _chunk_cuts(off, n_chunks):
    """The read boundaries of hx_chunk_end (hx_internal.cuh): chunk c ends at the first read whose offset reaches
    off[0] + (c + 1) / n_chunks of the alleles."""
    R = len(off) - 1
    n = int(off[-1] - off[0])
    n_chunks = min(n_chunks, R)
    cuts = [0]
    for c in range(n_chunks - 1):
        a = cuts[-1]
        cuts.append(a + int(np.searchsorted(off[a:R], off[0] + n * (c + 1) // n_chunks, side="left")))
    return cuts + [R]


def _pipeline_chunks(off, slim=True):
    n = int(off[-1] - off[0])
    return max(6 if slim else 3, -(-n // CHUNK_CODES))


def _oracle(c_oracle, rank, off, codes, N, W):
    ref, rt = c_oracle.ingest(rank, off, codes, N, W)
    return dict(rank=rank, off=off, codes=codes, N=N, W=W, ref=ref.astype(np.float32), rt=_totals(rt))


def _new(c):
    from gretel_b200.hansel import Hansel, REF_SYMBOLS, REF_UNSYMBOLS
    return Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, c["N"], band_w=c["W"])


def _check(h, totals, want_rt, want_ref, what):
    band = h.band()
    h.close()
    assert totals == want_rt, what
    _assert_band(band, want_ref, what)


def _host(c, what, h=None):
    """hx_ingest_host of the whole case into a new matrix, compared with the oracle."""
    h = h or _new(c)
    _check(h, h.ingest_packed(c["rank"], c["off"], c["codes"]), c["rt"], c["ref"], what)


def _dense(c, what):
    """One hx_ingest_host_dense call (the numpy encoder) into a new matrix, compared with the oracle."""
    from gretel_b200 import util
    h = _new(c)
    _check(h, h.ingest_packed_dense(util.dense_packed(c["rank"], c["off"], c["codes"])), c["rt"], c["ref"], what)


def _compact(c, what):
    from gretel_b200 import util
    h = _new(c)
    klen, codes4, n_codes = util.compact_packed(c["off"], c["codes"])
    _check(h, h.ingest_packed_compact(c["rank"], klen, codes4, n_codes), c["rt"], c["ref"], what)


def _env(monkeypatch, **kv):
    for key, v in kv.items():
        if v is None:
            monkeypatch.delenv(key, raising=False)
        else:
            monkeypatch.setenv(key, str(v))


# ---- 1. the spine's carry from one step of 1024 blocks to the next ----------------------------------------------------

def _carry_input(R, wide, seed):
    """R reads of 0-4 SNPs.  Escapes (rank gaps >= 255, one of exactly 255) sit at read 0 and inside every spine step,
    at the last read of the first step and the first of the second, and at the last read (a gap of 300, so that the
    chunk's last escape differs from the 255 its placeholder byte holds); about 5 % of the alleles are N / - / _.
    wide: one read of 256 SNPs (uint16 SNP counts, W = 255) in the last step."""
    rng = np.random.default_rng(seed)
    k = rng.integers(0, 5, size=R, dtype=np.int64)
    d = np.zeros(R, np.int64)
    _steps(rng, d, 400)
    esc = {0: 300, 16: 255, 4096 * 700 + 15: 256, SPINE_STEP - 1: 400, SPINE_STEP: 257, SPINE_STEP + 16: 255,
           2 * SPINE_STEP - 1: 270, 2 * SPINE_STEP + 4095: 256, R - 1: 300}
    for i, gap in esc.items():
        if i < R:
            d[i] = gap
            k[i] = max(k[i], 2)
    if wide:
        k[R - 3] = 256
    W = 255 if wide else 3
    rank, off, codes, N = _reads(k, d, rng)
    return rank, off, codes, N, W


@pytest.mark.parametrize("wide", [False, True], ids=["klen8", "klen16"])
@pytest.mark.parametrize("n_reads", [SPINE_STEP - 1, SPINE_STEP, SPINE_STEP + 1, 9_000_000])
def test_dense_chunk_spine_carry(c_oracle, n_reads, wide):
    """One ingest_packed_dense chunk around the spine's step: nblk = (n + 1 + 4095) / 4096 is 1024 at n = 4,194,303
    (one step), 1025 at 4,194,304 (the second step holds off[n] alone) and at 4,194,305 (one read and off[n]), and
    2198 at 9M reads (three steps).  Ranks, offsets and run ends of the later steps rest on the carry."""
    from gretel_b200 import util
    c = _oracle(c_oracle, *_carry_input(n_reads, wide, n_reads % 1000 + wide))
    dense = util.dense_packed(c["rank"], c["off"], c["codes"])
    assert dense.klen.dtype == (np.uint16 if wide else np.uint8)
    assert len(dense.esc_idx) >= 4 and dense.esc_delta[-1] != 255
    assert len(dense.exc_pos) > 0 and (-(-(n_reads + 1) // 4096) > 1024) == (n_reads >= SPINE_STEP)
    h = _new(c)
    _check(h, h.ingest_packed_dense(dense), c["rt"], c["ref"], "dense chunk of %d reads, W=%d" % (n_reads, c["W"]))


@pytest.mark.parametrize("W", [3, 255])
def test_host_pipeline_chunks_past_one_spine_step(c_oracle, monkeypatch, W):
    """The default hx_ingest_host on 26.5M reads of 2-3 SNPs: six slim chunks of more than 4,194,304 reads each, so
    every chunk's spine takes a second step.  Escapes at each chunk's first read, first read of the second step and last
    read.  W = 255 selects uint16 SNP counts from the band (and one read of 256 SNPs uses it)."""
    _env(monkeypatch, HX_HOST_PIPELINE=None, HX_HOST_THREADS=None)
    rng = np.random.default_rng(26 + W)
    R = 26_500_000
    k = rng.integers(2, 4, size=R, dtype=np.int64)
    if W == 255:
        k[R // 2] = 256
    off = np.zeros(R + 1, np.int64)
    np.cumsum(k, out=off[1:])
    cuts = _chunk_cuts(off, _pipeline_chunks(off))
    assert len(cuts) == 7 and min(np.diff(cuts)) > SPINE_STEP
    d = np.zeros(R, np.int64)
    _steps(rng, d, 400)
    for a, b in zip(cuts[:-1], cuts[1:]):
        d[a + SPINE_STEP] = 256
        d[b - 1] = 300
    del off
    c = _oracle(c_oracle, *_reads(k, d, rng), W)
    del k, d
    _host(c, "slim pipeline, 26.5M reads, W=%d" % W)


# ---- 2. escapes and rank runs on the decode granules -----------------------------------------------------------------

_ESC_AT = (15, 16, 17, 31, 32, 4095, 4096, 4097, 4111, 4112, 8191, 8192)
_ESC_GAPS = (255, 256, 300, 255, 511, 1000)
_STEP_AT = (1, 14, 15, 16, 47, 48, 63, 4080, 4094, 4095, 4096, 4098, 8190, 8192)


def _granule_input(R, seed, n_chunks=1, first_escape=True, last="escape"):
    """Reads placed on the granules of every chunk (the cuts of _chunk_cuts): escapes at chunk-relative reads that are
    15, 0 and 16 mod 16 and 4095, 4096 mod 4096, so that the read after a thread's 16 (what k_dense_apply looks up for
    the end of its last run) is an escape; gaps of exactly 255 among them.  Rank steps of 1 start and end runs on the
    same boundaries.  The chunk's last read is an escape of 300 (the last entry of its escape list), or last="run":
    the last 20 reads share one rank.  Reads of 0-12 SNPs, at least 2 where something is placed; in several chunks
    2-11 everywhere, so that the cuts do not move.  The allele count is not a multiple of 4 (nor of 16)."""
    rng = np.random.default_rng(seed)
    k = rng.integers(0 if n_chunks == 1 else 2, 12, size=R, dtype=np.int64)
    if k.sum() % 4 == 0:
        k[0] = 2 if k[0] != 2 else 3
    off = np.zeros(R + 1, np.int64)
    np.cumsum(k, out=off[1:])
    cuts = _chunk_cuts(off, n_chunks)
    d = np.zeros(R, np.int64)
    _steps(rng, d, max(1, R // 10))
    for a, b in zip(cuts[:-1], cuts[1:]):
        placed = [(a + rel, 1) for rel in _STEP_AT] + [(a + rel, _ESC_GAPS[j % len(_ESC_GAPS)])
                                                        for j, rel in enumerate(_ESC_AT)]
        for i, gap in placed:
            if i < b:
                d[i] = gap
                k[i] = max(k[i], 2)
        if last == "escape":
            d[b - 1] = 300
        else:
            d[max(a + 1, b - 19):b] = 0
            d[max(a + 1, b - 20)] = 1
        k[b - 2:b] = np.maximum(k[b - 2:b], 2)
    d[0] = 400 if first_escape else 0
    if k.sum() % 4 == 0:                         # single chunk: the forced widths moved the count
        k[R - 1] += 1
    assert k.sum() % 4 and (n_chunks == 1 or _chunk_cuts(np.concatenate([[0], np.cumsum(k)]), n_chunks) == cuts)
    rank, off, codes, N = _reads(k, d, rng, p_special=0.2, pad=2)
    return rank, off, codes, N, 11


_GRANULE_CASES = [(R, first, last) for R in (15, 16, 17, 4095, 4096, 4097)
                  for first, last in ((True, "escape"), (False, "run"))]


@pytest.mark.parametrize("R,first_escape,last", _GRANULE_CASES)
@pytest.mark.parametrize("path", ["dense", "compact"])
def test_decode_granules(c_oracle, path, R, first_escape, last):
    """n_reads of 15, 16, 17, 4095, 4096 and 4097 (off[n] in a block of its own at 4096), hand-placed escapes and runs,
    through ingest_packed_dense and the compact path."""
    c = _case(c_oracle, "wire-granules-%d-%d-%s" % (R, first_escape, last),
              lambda: _granule_input(R, R + 7 * first_escape, first_escape=first_escape, last=last))
    what = "%s, %d reads, first read %s, last %s" % (path, R, "escape" if first_escape else "rank 0", last)
    (_dense if path == "dense" else _compact)(c, what)


@pytest.mark.parametrize("pipeline", ["slim", "dense"])
@pytest.mark.parametrize("last", ["escape", "run"])
def test_pipeline_chunk_granules(c_oracle, monkeypatch, pipeline, last):
    """The same granules relative to every chunk the slim pipeline cuts 230k reads into (the dense pipeline's three
    chunks start where slim chunks 0, 2 and 4 do); chunks after the first start with an escape of their absolute rank."""
    _env(monkeypatch, HX_HOST_PIPELINE=pipeline, HX_HOST_THREADS=3)
    R = 230_000
    c = _case(c_oracle, "wire-pipeline-granules-%s" % last, lambda: _granule_input(R, 230 + (last == "run"), 6,
                                                                                   last=last))
    assert R >= PIPELINE_MIN_READS and _pipeline_chunks(c["off"]) == 6
    _host(c, "%s pipeline, granules in every chunk, last %s" % (pipeline, last))


# ---- 3. pinned slots and staging sets that grow while other chunks are in flight ---------------------------------------

def _segments(seed, parts, W=3):
    """Rank-sorted reads in consecutive segments of (reads, kmin, kmax, p_special); escapes inside each."""
    rng = np.random.default_rng(seed)
    ks, ps = [], []
    for n, lo, hi, p in parts:
        ks.append(rng.integers(lo, hi + 1, size=n, dtype=np.int64))
        ps.append(p)
    k = np.concatenate(ks)
    d = np.zeros(len(k), np.int64)
    _steps(rng, d, 500)
    d[rng.integers(1, len(k), size=2 * len(parts))] = 260
    rank = np.cumsum(d)
    N = int((rank + k).max())
    off = np.zeros(len(k) + 1, np.int64)
    np.cumsum(k, out=off[1:])
    codes = np.concatenate([_codes(rng, int(x.sum()), p) for x, p in zip(ks, ps)])
    bounds = np.cumsum([0] + [n for n, *_ in parts])
    return rank.astype(np.int32), off, codes, N, W, bounds


def test_dense_chunks_grow_staging_in_flight(c_oracle):
    """Five ingest_packed_dense chunks enqueued with wait=False: the last ones hold 2.5-3x the reads and 6-15x the
    exceptions of the first, so the staging sets grow while the earlier chunks are still being decoded and expanded."""
    from gretel_b200 import util
    parts = [(20_000, 0, 4, 0.02), (20_000, 0, 4, 0.02), (30_000, 0, 4, 0.1), (50_000, 0, 4, 0.2), (60_000, 0, 4, 0.3)]
    rank, off, codes, N, W, bounds = _segments(31, parts)
    c = _oracle(c_oracle, rank, off, codes, N, W)
    chunks = [util.dense_packed(rank[a:b], off[a:b + 1], codes) for a, b in zip(bounds[:-1], bounds[1:])]
    assert chunks[-1].n_reads >= 2.5 * chunks[0].n_reads and len(chunks[-1].exc_pos) >= 6 * len(chunks[0].exc_pos)
    h = _new(c)
    for ch in chunks:
        assert h.ingest_packed_dense(ch, wait=False) is None
    _check(h, h.ingest_totals(), c["rt"], c["ref"], "five growing dense chunks")


@pytest.mark.parametrize("pipeline", ["slim", "dense"])
def test_pipeline_grows_slots_and_sets_mid_input(c_oracle, monkeypatch, pipeline):
    """Wide reads (20-29 SNPs, 5 % exceptions) for the first half of the alleles, then 2-3 SNP reads with 60 %
    exceptions: the last chunk holds about ten times the reads of the first (staging sets grow) and, in the dense pipeline,
    exception lists larger than the pinned slot's headroom (the slot grows keeping the bytes already encoded)."""
    _env(monkeypatch, HX_HOST_PIPELINE=pipeline, HX_HOST_THREADS=3)
    c = _case(c_oracle, "wire-wide-then-narrow", lambda: _segments(
        32, [(80_000, 20, 29, 0.05), (800_000, 2, 3, 0.6)], W=28)[:5])
    cuts = _chunk_cuts(c["off"], _pipeline_chunks(c["off"], pipeline == "slim"))
    assert np.diff(cuts)[-1] >= 8 * np.diff(cuts)[0]
    _host(c, "%s pipeline, wide reads then narrow exception-dense reads" % pipeline)


def _pipelined(c_oracle, name, R, W, kmax, seed, N=5000):
    """R reads of 0-kmax SNPs over N sites, 10 % N / - / _, rank steps at N / 4 reads and four escapes."""
    def make():
        rng = np.random.default_rng(seed)
        k = rng.integers(0, kmax + 1, size=R, dtype=np.int64)
        d = np.zeros(R, np.int64)
        _steps(rng, d, N // 4)
        d[rng.integers(1, R, size=4)] = 255 + rng.integers(0, 50, size=4)
        rank, off, codes, N_ = _reads(k, d, rng, p_special=0.1, N=N)
        return rank, off, codes, N_, W
    return _case(c_oracle, name, make)


@pytest.mark.parametrize("pipeline", ["slim", "dense"])
def test_second_larger_ingestion_adds(c_oracle, monkeypatch, pipeline):
    """ingest_packed of 250k reads, then of 600k reads into the same matrix: the second call's chunks are larger than
    every buffer the first sized, and the counts and totals add."""
    _env(monkeypatch, HX_HOST_PIPELINE=pipeline, HX_HOST_THREADS=None)
    a = _pipelined(c_oracle, "wire-250k", 250_000, 7, 8, 41)
    b = _pipelined(c_oracle, "wire-600k", 600_000, 7, 8, 42)
    h = _new(a)
    assert h.ingest_packed(a["rank"], a["off"], a["codes"]) == a["rt"]
    _check(h, h.ingest_packed(b["rank"], b["off"], b["codes"]), _add(a["rt"], b["rt"]), a["ref"] + b["ref"],
           "%s pipeline, 250k then 600k reads" % pipeline)


@pytest.mark.parametrize("pipeline", ["slim", "dense"])
def test_two_matrices_alternate_on_one_thread(c_oracle, monkeypatch, pipeline):
    """The encoder's plan is one per host thread: two matrices fed alternately from this thread, one with uint8 SNP
    counts (W = 7), one with uint16 (W = 300, reads of up to 32 SNPs), each in two halves of at least 200k reads."""
    _env(monkeypatch, HX_HOST_PIPELINE=pipeline, HX_HOST_THREADS=None)
    a = _pipelined(c_oracle, "wire-500k", 500_000, 7, 8, 43)
    b = _pipelined(c_oracle, "wire-w300-400k", 400_000, 300, 32, 44, N=2000)
    ha, hb = _new(a), _new(b)
    half = lambda h, x, lo, hi: h.ingest_packed(x["rank"][lo:hi], x["off"][lo:hi + 1], x["codes"])
    Ra, Rb = len(a["rank"]), len(b["rank"])
    half(ha, a, 0, Ra // 2)
    half(hb, b, 0, Rb // 2)
    ta = half(ha, a, Ra // 2, Ra)
    tb = half(hb, b, Rb // 2, Rb)
    _check(ha, ta, a["rt"], a["ref"], "%s pipeline, matrix A (W=7) alternating with B" % pipeline)
    _check(hb, tb, b["rt"], b["ref"], "%s pipeline, matrix B (W=300) alternating with A" % pipeline)


# ---- 4. pipeline shapes ---------------------------------------------------------------------------------------------

def test_pipeline_more_than_six_chunks(c_oracle, monkeypatch):
    """25.5M reads of mostly 8 SNPs: 6 * 32 Mi alleles and more, so the slim pipeline cuts seven chunks."""
    _env(monkeypatch, HX_HOST_PIPELINE=None, HX_HOST_THREADS=None)
    rng = np.random.default_rng(7)
    R = 25_500_000
    k = np.full(R, 8, np.int64)
    few = rng.integers(0, R, size=R // 100)
    k[few] = rng.integers(0, 8, size=len(few))
    d = np.zeros(R, np.int64)
    _steps(rng, d, 1500)
    d[rng.integers(1, R, size=14)] = 300
    c = _oracle(c_oracle, *_reads(k, d, rng), 7)
    del k, d
    assert 6 * CHUNK_CODES < len(c["codes"]) and _pipeline_chunks(c["off"]) == 7
    _host(c, "slim pipeline, 7 chunks")


@pytest.mark.parametrize("threads", [1, 3, None], ids=["threads1", "threads3", "threads-default"])
@pytest.mark.parametrize("pipeline", [None, "dense", "packed", "off"], ids=["default", "dense", "packed", "off"])
def test_pipeline_and_thread_knobs(c_oracle, monkeypatch, pipeline, threads):
    """HX_HOST_PIPELINE x HX_HOST_THREADS on 320k reads with escapes and exceptions: every setting equals the oracle."""
    _env(monkeypatch, HX_HOST_PIPELINE=pipeline, HX_HOST_THREADS=threads)
    _host(_pipelined(c_oracle, "wire-320k", 320_000, 11, 12, 45), "HX_HOST_PIPELINE=%s HX_HOST_THREADS=%s"
          % (pipeline, threads))


@pytest.mark.parametrize("pipeline", ["slim", "dense"])
def test_pipeline_uint16_counts_from_the_band(c_oracle, monkeypatch, pipeline):
    """W = 300 with reads of at most 32 SNPs: the pipeline takes its SNP-count width from W + 1 >= 256, not from the
    reads, and ships uint16 counts of short reads."""
    _env(monkeypatch, HX_HOST_PIPELINE=pipeline, HX_HOST_THREADS=None)
    c = _pipelined(c_oracle, "wire-w300-400k", 400_000, 300, 32, 44, N=2000)
    assert int(np.diff(c["off"]).max()) <= 32
    _host(c, "%s pipeline, W=300, reads of <= 32 SNPs" % pipeline)


@pytest.mark.parametrize("pipeline", ["slim", "dense", "packed"])
def test_pipeline_shard_slices(c_oracle, monkeypatch, pipeline):
    """rank[a:b], off[a:b+1] (absolute offsets, off[0] != 0) and the whole codes array, as the multi-GPU loader passes
    its shard, for three shards of at least 200k reads ingested into one matrix: the sum is the oracle's whole band."""
    from gretel_b200 import dist
    _env(monkeypatch, HX_HOST_PIPELINE=pipeline, HX_HOST_THREADS=None)
    c = _pipelined(c_oracle, "wire-700k", 700_000, 11, 12, 46)
    bounds = dist.shard_bounds(c["off"], 3)
    assert min(np.diff(bounds)) >= PIPELINE_MIN_READS
    h = _new(c)
    for a, b in zip(bounds[:-1], bounds[1:]):
        a, b = int(a), int(b)
        assert a == 0 or c["off"][a] != 0
        totals = h.ingest_packed(c["rank"][a:b], c["off"][a:b + 1], c["codes"])
    _check(h, totals, c["rt"], c["ref"], "%s pipeline, three shards" % pipeline)


# ---- 5. the compact path's scan --------------------------------------------------------------------------------------

@pytest.mark.parametrize("R", [4094, 4095, 4096, 3 * 4096 - 1])
def test_compact_scan_blocks(c_oracle, R):
    """hx_ingest_host_compact scans n_reads + 1 = 4095, 4096, 4097 and 3 * 4096 SNP counts (blocks of 4096), some of
    them above 255 (W = 299), with an odd allele count."""
    def make():
        rng = np.random.default_rng(R)
        k = rng.integers(0, 20, size=R, dtype=np.int64)
        k[rng.integers(0, R, size=6)] = rng.integers(256, 301, size=6)
        k[-1] = 256
        if k.sum() % 2 == 0:
            k[-1] = 257
        d = np.zeros(R, np.int64)
        _steps(rng, d, 300)
        d[R // 3] = 255
        rank, off, codes, N = _reads(k, d, rng, p_special=0.1)
        return rank, off, codes, N, 299
    c = _case(c_oracle, "wire-compact-%d" % R, make)
    assert len(c["codes"]) % 2 == 1 and int(np.diff(c["off"]).max()) > 255
    _compact(c, "compact path, %d reads" % R)


# ---- 6. bad reads: one status at every size and under every pipeline --------------------------------------------------

_BAD = ("wider_than_band", "over_255_snps", "code_7")


def _bad_input(R, bad):
    """R reads of 2-8 SNPs in a band of W = 29; read 3R/5 (a later chunk of the pipelines) is bad: 31 SNPs (wider than
    the band), 256 SNPs (more than a uint8 SNP count; the band's W + 1 < 256 selects that width), or allele code 7;
    bad="valid": none of them.  N = 3100."""
    rng = np.random.default_rng(R + len(bad))
    k = rng.integers(2, 9, size=R, dtype=np.int64)
    i = 3 * R // 5
    if bad in ("wider_than_band", "over_255_snps"):
        k[i] = 31 if bad == "wider_than_band" else 256
    d = np.zeros(R, np.int64)
    _steps(rng, d, 1000)
    d[i + 1:i + 3] = 255
    rank, off, codes, N = _reads(k, d, rng, N=3100)
    if bad == "code_7":
        codes[off[i] + 1] = 7
    return rank, off, codes, N, 29


_BAD_INPUTS = {}


def _bad(R, bad):
    if (R, bad) not in _BAD_INPUTS:
        _BAD_INPUTS[(R, bad)] = _bad_input(R, bad)
    return _BAD_INPUTS[(R, bad)]


def _valid_after_reset(c_oracle, h):
    """After the refusal, reset_counts() and a valid input gives the oracle's band and totals bit for bit."""
    c = _case(c_oracle, "wire-valid-after-refusal", lambda: _bad_input(3000, "valid"))
    h.reset_counts()
    _check(h, h.ingest_packed(c["rank"], c["off"], c["codes"]), c["rt"], c["ref"], "valid input after a refusal")


@pytest.mark.parametrize("bad", _BAD)
@pytest.mark.parametrize("pipeline", [None, "slim", "dense", "packed", "off"],
                         ids=["default", "slim", "dense", "packed", "off"])
def test_bad_reads_refused_alike(c_oracle, monkeypatch, pipeline, bad):
    """The same bad read in 5000 reads (one launch) and in 250k reads (the pipeline, when HX_HOST_PIPELINE selects
    one): hx_ingest_host returns HX_E_READ for both."""
    from gretel_b200 import _lib
    from gretel_b200.hansel import Hansel, REF_SYMBOLS, REF_UNSYMBOLS
    _env(monkeypatch, HX_HOST_PIPELINE=pipeline, HX_HOST_THREADS=None)
    for R in (5000, 250_000):
        rank, off, codes, N, W = _bad(R, bad)
        h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=W)
        with pytest.raises(_lib.HanselxError) as e:
            h.ingest_packed(rank, off, codes)
        assert e.value.code == _lib.HX_E_READ, (R, pipeline, bad, str(e.value))
        _valid_after_reset(c_oracle, h)


@pytest.mark.parametrize("bad", _BAD)
def test_bad_reads_refused_alike_dense_wire(c_oracle, bad):
    """The same bad reads through ingest_packed_dense, at 5000 and 250k reads: the wide reads travel with uint16 SNP
    counts, code 7 as a 2-bit field of 3 at an exception position.  HX_E_READ for all."""
    from gretel_b200 import _lib, util
    from gretel_b200.hansel import Hansel, REF_SYMBOLS, REF_UNSYMBOLS
    for R in (5000, 250_000):
        rank, off, codes, N, W = _bad(R, bad)
        if bad == "code_7":
            p = int(np.flatnonzero(codes == 7)[0])
            codes = codes.copy()
            codes[p] = 6
        dense = util.dense_packed(rank, off, codes)
        if bad == "code_7":
            dense.codes2[p >> 2] |= 3 << (2 * (p & 3))
        h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=W)
        with pytest.raises(_lib.HanselxError) as e:
            h.ingest_packed_dense(dense)
        assert e.value.code == _lib.HX_E_READ, (R, bad, str(e.value))
        _valid_after_reset(c_oracle, h)
