"""Ingestion under the launch conditions production reaches beyond a fresh matrix on a whole GPU: reduced SM budgets
(the overlapped multi-GPU step leaves SMs to the collective), counts on top of counts (the read-modify-write epilogues,
counts written by the caller, a matrix taken back from the parking lot), shard slices through the device entry point,
the CTA-pair long-read kernel and the slice-weight overrides.  Every result is compared with the C oracle: the float32
band bit for bit and all four totals."""
import os
import subprocess
import sys

import numpy as np
import pytest

from gretel_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- helpers -----------------------------------------------------------------------------------------------------

def _new(N, W, kernel, sms=None):
    from gretel_b200.hansel import Hansel, REF_SYMBOLS, REF_UNSYMBOLS
    h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=W)
    h.set_ingest_kernel(kernel)
    if sms is not None:
        h.set_ingest_sms(sms)
    return h


def _assert_band(band, want, what):
    """Bit-exact band; on a mismatch, the first cells that differ (band row pj, distance d, symbols a, b)."""
    if np.array_equal(band, want):
        return
    bad = np.argwhere(band != want)
    cells = ["pj=%d d=%d a=%d b=%d got %g want %g" % (i[0], i[1] + 1, i[2], i[3], band[tuple(i)], want[tuple(i)])
             for i in bad[:12]]
    pytest.fail("%s: %d cells differ\n    %s" % (what, len(bad), "\n    ".join(cells)))


def _totals(rt):
    return tuple(int(x) for x in rt)


def _add(*rts):
    return tuple(int(sum(x)) for x in zip(*rts))


def _pack(rank, k, rng, p_special=0.05):
    """Rank-sorted packed reads of k[i] SNPs at rank[i], random alleles (a few N / - / _)."""
    order = np.argsort(rank, kind="stable")
    rank, k = np.asarray(rank)[order].astype(np.int32), np.asarray(k)[order].astype(np.int64)
    off = np.concatenate([[0], np.cumsum(k)]).astype(np.int64)
    codes = rng.integers(0, 4, size=int(off[-1])).astype(np.uint8)
    sp = rng.random(len(codes)) < p_special
    codes[sp] = rng.integers(4, 7, size=int(sp.sum())).astype(np.uint8)
    return rank, off, codes


def _skewed(shape):
    """The skewed shapes of test_gpu_ingest.test_slices_and_job_tables_on_skewed_shapes."""
    rng = np.random.default_rng({"one_run": 1, "many_runs_per_cta": 2, "mostly_narrow_reads": 3, "rank_jumps": 4,
                                 "dense_then_sparse": 5}[shape])
    if shape == "one_run":
        N, R = 40, 300_000
        rank = np.full(R, 5)
        k = rng.integers(2, 21, size=R)
    elif shape == "many_runs_per_cta":
        N, R = 300_000, 150_000                  # ~118k populated ranks
        rank = rng.integers(0, N - 8, size=R)
        k = rng.integers(2, 9, size=R)
    elif shape == "mostly_narrow_reads":
        N, R = 2000, 250_000
        rank = rng.integers(0, N - 12, size=R)
        k = np.where(rng.random(R) < 0.9, rng.integers(0, 2, size=R), rng.integers(2, 13, size=R))
    elif shape == "rank_jumps":
        N, R = 50_000, 120_000
        rank = rng.choice(np.arange(0, N - 32, 977), size=R)      # 52 populated ranks, 977 apart
        k = rng.integers(2, 31, size=R)
    else:
        N, R = 6000, 200_000
        dense = rng.random(R) < 0.8
        rank = np.where(dense, rng.integers(0, 300, size=R), rng.integers(300, N - 30, size=R))
        k = np.where(dense, rng.integers(20, 31, size=R), rng.integers(2, 6, size=R))
    k = np.minimum(k, N - rank)
    rank, off, codes = _pack(rank, k, rng, p_special=0.02)
    return rank, off, codes, N, int(max(1, k.max() - 1))


def _workload(name, n_reads):
    d = synth.generate(synth.scaled(synth.WORKLOADS[name], n_reads))
    return d["rank"], d["off"], d["codes"], d["n_snps"], d["max_k"] - 1


def _unsorted(seed, N, R, mk):
    rank, off, codes = synth.random_packed(np.random.default_rng(seed), N, R, mk, p_special=0.1, sort=False)
    return rank, off, codes, N, mk - 1


def _random_seed(seed):
    """The inputs of test_gpu_ingest.test_random_packed_bit_exact."""
    rng = np.random.default_rng(500 + seed)
    N = int(rng.integers(2, 200))
    R = int(rng.integers(1, 3000))
    mk = int(rng.integers(2, 40))
    rank, off, codes = synth.random_packed(rng, N, R, mk, p_special=0.2, sort=bool(seed % 2))
    W = max(1, min(mk, N) - 1) if seed % 3 else min(N + 1, 64)
    return rank, off, codes, N, W


_EDGES = [   # the inputs of test_gpu_ingest.test_edge_cases
    (np.zeros(0, np.int32), np.zeros(1, np.int64), np.zeros(0, np.uint8), 5, 3),
    (np.array([0, 1, 2], np.int32), np.array([0, 1, 1, 2], np.int64), np.array([0, 1], np.uint8), 5, 3),
    (np.array([0, 0], np.int32), np.array([0, 2, 4], np.int64), np.array([0, 1, 4, 2], np.uint8), 2, 1),
    (np.array([0, 2, 3], np.int32), np.array([0, 5, 8, 10], np.int64),
     np.array([0, 1, 2, 3, 5, 6, 0, 4, 4, 1], np.uint8), 5, 4),
]

_SHAPES = {
    "config3": lambda: _workload("metagenome", 150_000),     # configs[2] scaled: N = 10k, W = 29
    "many_runs_per_cta": lambda: _skewed("many_runs_per_cta"),
    "rank_jumps": lambda: _skewed("rank_jumps"),
    "ont": lambda: _workload("ont", 300),                     # N = 10k, W = 587
    "mid": lambda: _workload("mid", 20_000),                  # 80 SNPs per read, N = 10k, W = 110
    "unsorted_random": lambda: _unsorted(7, 3000, 40_000, 24),
    "unsorted_short": lambda: _unsorted(8, 3000, 100_000, 24),   # < 64 (N + 1): auto picks the bit-sliced kernel
    # for the slices of the device entry: short reads over 10k sites, 80-SNP reads over 1000 sites
    "short_slices": lambda: _workload("metagenome", 60_000),
    "long_slices": lambda: (lambda d: (d["rank"], d["off"], d["codes"], d["n_snps"], d["max_k"] - 1))(
        synth.generate(synth.Workload("mid-1k", 2, 10_000, 1_000, 6_000, 800, 0.005, 0.001))),
}
_SHAPES.update({"skewed_" + s: (lambda s=s: _skewed(s))
                for s in ("one_run", "many_runs_per_cta", "mostly_narrow_reads", "rank_jumps", "dense_then_sparse")})
_SHAPES.update({"seed%d" % s: (lambda s=s: _random_seed(s)) for s in range(8)})
_SHAPES.update({"edge%d" % i: (lambda i=i: _EDGES[i]) for i in range(len(_EDGES))})

_ORACLE = {}


def _case(c_oracle, name, make=None):
    """Inputs and the C oracle's band (float32: every count here is far below 2^24) and totals, once per process."""
    if name not in _ORACLE:
        rank, off, codes, N, W = (make or _SHAPES[name])()
        ref, rt = c_oracle.ingest(rank, off, codes, N, W)
        _ORACLE[name] = dict(rank=rank, off=off, codes=codes, N=N, W=W, ref=ref.astype(np.float32), rt=_totals(rt))
    return _ORACLE[name]


def _ingest(c, kernel, sms=None):
    h = _new(c["N"], c["W"], kernel, sms)
    totals = h.ingest_packed(c["rank"], c["off"], c["codes"])
    band = h.band()
    h.close()
    return band, totals


# ---- 1. SM budgets --------------------------------------------------------------------------------------------------

_BUDGETS = (1, 2, 3, 5, 124, 147)
_SM_CASES = ([(k, s) for s in ("config3", "many_runs_per_cta", "rank_jumps") for k in (6, 2, 4, 5)] +
             [(k, s) for s in ("ont", "mid") for k in (7, 3)] + [(1, "unsorted_random"), (0, "unsorted_short")])


@pytest.mark.parametrize("kernel,shape", _SM_CASES)
def test_sm_budget(c_oracle, kernel, shape):
    """set_ingest_sms(n) for n in 1, 2, 3, 5, 124, 147, then 0 again (all SMs).  Each shape has fewer than 200k reads, so
    one ingest_packed is one launch, and enough reads that the budget, not the one-CTA-per-256-reads clamp, sets the grid:
    - sorted-run kernels (2, 4, 5 bit-sliced; 6 tensor-core): grid = min(n * occ, ceil(R / 256)) with occ <= 2 CTAs per
      SM, and ceil(R / 256) >= 391 > 2 * 147 (asserted), so grid = n * occ: one or two CTAs hold every read at n = 1.
      k1_umma sizes its job tables from that grid: at n = 1 the "many runs per CTA" shape puts ~118k runs (~460
      batches of 256) and the "rank jumps" shape runs 977 ranks apart into one CTA.
    - 7 (k_l2_tiles): grid = n directly.  3 (bit-plane tiles): its tile grid follows the geometry, not the budget; only
      its idle unsorted-input fallback (k1_pairs_red) is sized by it.
    - 1 (k1_pairs_red): grid = min(ceil(R / 8), 8 n) = 8 n, as ceil(R / 8) = 5000 > 8 * 147.
    - 0 (auto) on unsorted short reads: the bit-sliced kernel (grid n * occ) declines and the fallback queued behind it
      runs.  A first ingestion of the same reads makes this process meet unsorted input, so that fallback is the
      counting-sort tensor-core kernel, k_l2_tiles with grid = n."""
    c = _case(c_oracle, shape)
    R = len(c["rank"])
    assert R < 200_000
    if kernel in (2, 4, 5, 6, 0):
        assert (R + 255) // 256 > 2 * max(_BUDGETS)
    if kernel == 1:
        assert (R + 7) // 8 > 8 * max(_BUDGETS)
    if kernel == 0:
        band, totals = _ingest(c, 0)
        assert totals == c["rt"]
    for n in _BUDGETS + (0,):
        h = _new(c["N"], c["W"], kernel)
        if n == 0:
            h.set_ingest_sms(5)
        h.set_ingest_sms(n)
        totals = h.ingest_packed(c["rank"], c["off"], c["codes"])
        band = h.band()
        h.close()
        assert totals == c["rt"], "kernel %d, %s, %d SMs" % (kernel, shape, n)
        _assert_band(band, c["ref"], "kernel %d, %s, %d SMs" % (kernel, shape, n))


# ---- 2. counts on top of counts ------------------------------------------------------------------------------------

# (N, W): site blocks of 16 cut at 15 / 16 / 17 / 33 sites, W not a multiple of 16, and W = N + 1
_GEOMS = [(2, 1), (2, 3), (15, 7), (15, 16), (16, 9), (16, 17), (17, 13), (17, 18), (33, 21), (33, 34),
          (1007, 31), (1007, 1008)]
_KMAX = {6: 32, 5: 52, 2: 52}        # widest read (W + 1) the short-read kernels take; wider bands go elsewhere
_ON_TOP_KERNELS = (7, 3, 6, 5, 2, 1)


def _geoms(kernel):
    return [(N, W) for N, W in _GEOMS if W + 1 <= _KMAX.get(kernel, 1 << 30)]


def _irregular(N, W, seed):
    """Sorted reads over N sites in a band of W: reads at rank 0 (start sentinel), reads ending on site N (end
    sentinel), a read spanning all N sites where the band allows, some reads of 0 or 1 SNPs."""
    rng = np.random.default_rng(seed)
    R = 1500 if W < 100 else 300
    kmax = min(W + 1, N)
    k = rng.integers(2, kmax + 1, size=R)
    k[rng.random(R) < 0.05] = rng.integers(0, 2)
    rank = rng.integers(0, N - k + 1)
    rank[: R // 10] = 0
    rank[R // 10: R // 5] = N - k[R // 10: R // 5]
    if N <= W + 1:
        k[0], rank[0] = N, 0
    return _pack(rank, k, rng, p_special=0.1) + (N, W)


def _geom_case(c_oracle, N, W, seed):
    c = _case(c_oracle, "irregular-%d-%d-%d" % (N, W, seed), lambda: _irregular(N, W, seed))
    assert len(c["rank"]) > 0 and c["rt"][1] > 0 and c["rt"][3] > 0
    return c


@pytest.mark.parametrize("kernel", _ON_TOP_KERNELS)
def test_counts_on_top_of_counts(c_oracle, kernel):
    """Ingest A, then B into the same matrix: B lands on A's pending counts (A's ingestion turned the matrix's "fresh"
    state off, so kernel 7 takes its read-modify-write epilogue) and the result is oracle(A) + oracle(B)."""
    for N, W in _geoms(kernel):
        a, b = _geom_case(c_oracle, N, W, 1), _geom_case(c_oracle, N, W, 2)
        h = _new(N, W, kernel)
        assert h.ingest_packed(a["rank"], a["off"], a["codes"]) == a["rt"]
        totals = h.ingest_packed(b["rank"], b["off"], b["codes"])
        band = h.band()
        h.close()
        assert totals == _add(a["rt"], b["rt"]), (N, W)
        _assert_band(band, a["ref"] + b["ref"], "kernel %d, N=%d W=%d, A then B" % (kernel, N, W))


@pytest.mark.parametrize("kernel", _ON_TOP_KERNELS)
def test_counts_on_top_after_reset(c_oracle, kernel):
    """Ingest A, reset_counts(), ingest B: the counts are cleared and fresh again, the result is oracle(B) alone."""
    for N, W in _geoms(kernel):
        a, b = _geom_case(c_oracle, N, W, 1), _geom_case(c_oracle, N, W, 2)
        h = _new(N, W, kernel)
        h.ingest_packed(a["rank"], a["off"], a["codes"])
        h.reset_counts()
        totals = h.ingest_packed(b["rank"], b["off"], b["codes"])
        band = h.band()
        h.close()
        assert totals == b["rt"], (N, W)
        _assert_band(band, b["ref"], "kernel %d, N=%d W=%d, A, reset, B" % (kernel, N, W))


@pytest.mark.parametrize("kernel", _ON_TOP_KERNELS)
def test_counts_on_top_of_caller_writes(c_oracle, kernel):
    """include/hanselx.h: after the caller writes through hx_counts_buffer's pointer, the next ingestion adds to those
    counts.  A random pattern written there before the matrix's first ingestion must survive: pattern + oracle."""
    import torch
    from gretel_b200.dist import _DevBuf
    rng = np.random.default_rng(40 + kernel)
    for N, W in _geoms(kernel):
        a = _geom_case(c_oracle, N, W, 1)
        h = _new(N, W, kernel)
        ptr, n, _tptr, _tn = h.counts_buffer()
        assert n == (N + 2) * W * 49
        h.sync()                                               # the buffer was cleared on the matrix's stream
        pattern = rng.integers(0, 1 << 20, size=n, dtype=np.uint32)
        dev = torch.device("cuda", h.device)
        torch.as_tensor(_DevBuf(ptr, n, "<i4"), device=dev).copy_(torch.from_numpy(pattern.view(np.int32)))
        torch.cuda.synchronize(dev)
        totals = h.ingest_packed(a["rank"], a["off"], a["codes"])
        band = h.band()
        h.close()
        assert totals == a["rt"], (N, W)
        _assert_band(band, pattern.reshape(band.shape).astype(np.float32) + a["ref"],
                     "kernel %d, N=%d W=%d, on top of the caller's counts" % (kernel, N, W))


def test_counts_on_top_mixed_kernels(c_oracle):
    """Four ingestions into one matrix through different kernels - 6 (the first, into cleared counts), 7, 3, 1 - add up
    to the sum of the four oracles."""
    for N, W in _geoms(6):
        cases = [_geom_case(c_oracle, N, W, seed) for seed in (1, 2, 3, 4)]
        h = _new(N, W, 6)
        for kernel, c in zip((6, 7, 3, 1), cases):
            h.set_ingest_kernel(kernel)
            totals = h.ingest_packed(c["rank"], c["off"], c["codes"])
        band = h.band()
        h.close()
        assert totals == _add(*(c["rt"] for c in cases)), (N, W)
        _assert_band(band, sum(c["ref"] for c in cases), "N=%d W=%d, kernels 6, 7, 3, 1" % (N, W))


@pytest.mark.parametrize("finalized", [False, True], ids=["counts-pending", "band-folded"])
def test_counts_on_top_parked_matrix(c_oracle, finalized):
    """A destroyed matrix waits in the parking lot and the next one of its shape takes it back: whether it was destroyed
    with counts pending or after they were folded into the band, the new matrix's first ingestion (kernel 7, plain
    stores into cleared counts) gives oracle(B) alone."""
    if os.environ.get("HX_NO_MATRIX_CACHE"):
        pytest.skip("the matrix cache is disabled")
    N, W = 1007, 61                                    # a shape no other test here uses: the parked handle is ours
    a, b = _geom_case(c_oracle, N, W, 1), _geom_case(c_oracle, N, W, 2)
    h = _new(N, W, 7)
    h.ingest_packed(a["rank"], a["off"], a["codes"])
    if finalized:
        _assert_band(h.band(), a["ref"], "first matrix")
    handle = h._h.value
    h.close()
    h2 = _new(N, W, 7)
    assert h2._h.value == handle                       # taken back from the parking lot
    totals = h2.ingest_packed(b["rank"], b["off"], b["codes"])
    band = h2.band()
    h2.close()
    assert totals == b["rt"]
    _assert_band(band, b["ref"], "parked matrix, kernel 7")


# ---- 3. shard slices through the device entry point ---------------------------------------------------------------

@pytest.mark.parametrize("kernel", [0, 1, 2, 3, 5, 6, 7])
def test_device_entry_slices(c_oracle, kernel):
    """hx_ingest_device as the multi-GPU shards call it, on one GPU: the reads cut at shard_bounds for 2, 3 and 8 ranks,
    and once in the middle of the deepest rank's run; every slice passes rank[lo:hi] and the absolute offsets
    off[lo:hi+1] (neither starts at a 16-byte boundary) with the whole codes buffer, whose base sits at byte 0, 1 or 3
    of a padded allocation.  The slices of one cut add up to oracle(all reads), band and totals."""
    import torch
    from gretel_b200 import dist as gdist
    shapes = ["short_slices"] + (["long_slices"] if kernel in (0, 1, 3, 7) else [])
    dev = torch.device("cuda", 0)
    for shape in shapes:
        c = _case(c_oracle, shape)
        rank, off, codes = c["rank"], c["off"], c["codes"]
        R, n = len(rank), len(codes)
        runs = np.flatnonzero(np.diff(rank, prepend=-1, append=-1))          # first read of every run, and R
        deep = int(np.argmax(np.diff(runs)))
        mid = int(runs[deep] + runs[deep + 1]) // 2
        assert runs[deep] < mid < runs[deep + 1] and rank[mid - 1] == rank[mid]
        cuts = [gdist.shard_bounds(off, world) for world in (2, 3, 8)] + [np.array([0, mid, R])]
        t_rank = torch.from_numpy(rank).to(dev)
        t_off = torch.from_numpy(off).to(dev)
        for byte in (0, 1, 3):
            t_codes = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
            t_codes[byte:byte + n] = torch.from_numpy(codes).to(dev)
            torch.cuda.synchronize(dev)
            for bounds in cuts:
                h = _new(c["N"], c["W"], kernel)
                for lo, hi in zip(bounds[:-1], bounds[1:]):
                    lo, hi = int(lo), int(hi)
                    h.ingest_device(t_rank[lo:hi].data_ptr(), t_off[lo:hi + 1].data_ptr(), t_codes.data_ptr() + byte,
                                    hi - lo)
                totals = h.ingest_totals()
                band = h.band()
                h.close()
                what = "kernel %d, %s, codes at byte %d, cuts %s" % (kernel, shape, byte, list(bounds))
                assert totals == c["rt"], what
                _assert_band(band, c["ref"], what)


# ---- 4. knobs read once per process ---------------------------------------------------------------------------------

def _lumma_pairs(c_oracle):
    """Run in a process with HX_LUMMA_PAIRS=1 (see test_lumma_pairs)."""
    names = ["seed%d" % s for s in range(8)] + ["edge%d" % i for i in range(len(_EDGES))] + ["ont", "mid"]
    for name in names:
        c = _case(c_oracle, name)
        N, W = c["N"], c["W"]
        assert W // 16 + 2 <= 62                                   # g.SP: the pair kernel's limit
        launches = {}
        for sms in (0, 2, 3, 1):
            what = "%s (N=%d W=%d), %d SMs" % (name, N, W, sms)
            h = _new(N, W, 7, sms)
            before = h.launch_count()
            assert h.ingest_packed(c["rank"], c["off"], c["codes"]) == c["rt"], what
            launches[sms] = h.launch_count() - before
            _assert_band(h.band(), c["ref"], what + ", fresh")
            h.close()
            h = _new(N, W, 7, sms)
            h.ingest_packed(c["rank"], c["off"], c["codes"])
            assert h.ingest_packed(c["rank"], c["off"], c["codes"]) == _add(c["rt"], c["rt"]), what
            _assert_band(h.band(), 2 * c["ref"], what + ", on top")
            h.close()
        if len(c["rank"]):
            # the CTA-pair kernel counts one launch more than the single-CTA one it replaces: it ran at 2 SMs and
            # more, not at 1
            assert launches[2] == launches[3] == launches[0] == launches[1] + 1, (name, launches)
        print("pairs %s: N=%d W=%d ok" % (name, N, W))


def _slice_weights(c_oracle):
    """Run in a process with HX_UM_READ_W / HX_UM_RANK_W set (see test_slice_weights)."""
    for shape in ("one_run", "many_runs_per_cta", "mostly_narrow_reads", "rank_jumps", "dense_then_sparse"):
        c = _case(c_oracle, "skewed_" + shape)
        for kernel in (6, 2, 5):
            band, totals = _ingest(c, kernel)
            what = "%s, kernel %d, HX_UM_READ_W=%s HX_UM_RANK_W=%s" % (shape, kernel, os.environ.get("HX_UM_READ_W"),
                                                                       os.environ.get("HX_UM_RANK_W"))
            assert totals == c["rt"], what
            _assert_band(band, c["ref"], what)
        print("weights %s ok" % shape)


def _sorted_prefix(c_oracle):
    """Run in a fresh process (see test_sorted_prefix_unsorted_tail)."""
    def make():
        rank, off, codes, N, W = _workload("metagenome", 250_000)
        R = len(rank)
        head = R * 3 // 5
        perm = np.concatenate([np.arange(head), head + np.random.default_rng(2).permutation(R - head)])
        k = np.diff(off)
        off2 = np.concatenate([[0], np.cumsum(k[perm])]).astype(np.int64)
        idx = np.repeat(off[:-1][perm], k[perm]) + (np.arange(int(off2[-1])) - np.repeat(off2[:-1], k[perm]))
        return rank[perm], off2, codes[idx], N, W
    c = _case(c_oracle, "sorted_prefix", make)
    assert len(c["rank"]) >= 200_000 and not np.all(np.diff(c["rank"]) >= 0)
    launches = {}
    for step, kernel in (("first", 0), ("again", 0), ("fixed", 6)):
        h = _new(c["N"], c["W"], kernel)
        before = h.launch_count()
        totals = h.ingest_packed(c["rank"], c["off"], c["codes"])
        launches[step] = h.launch_count() - before
        band = h.band()
        h.close()
        assert totals == c["rt"], step
        _assert_band(band, c["ref"], "sorted prefix, unsorted tail, %s (kernel %d)" % (step, kernel))
    # the counting-sort fallback (12 launches per chunk of the tail) in both auto runs; one RED per pair (1 launch)
    # behind the fixed kernel
    assert launches["first"] == launches["again"] > launches["fixed"], launches
    print("sorted prefix ok: launches %s" % launches)


_SUB = r"""
import sys
from tests import test_gpu_ingest_launch as t
from oracle import c_oracle
getattr(t, sys.argv[1])(c_oracle)
"""


def _run_fresh(fn, **env):
    e = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), **env)
    e.pop("HX_HOST_PIPELINE", None)
    out = subprocess.run([sys.executable, "-c", _SUB, fn], capture_output=True, text=True, timeout=280, cwd=ROOT, env=e)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]


def test_lumma_pairs(c_oracle):
    """HX_LUMMA_PAIRS=1 (read once per process) turns on the CTA-pair long-read kernel k_l2_tiles2 (cta_group::2),
    launched on sms & ~1 CTAs when sms >= 2 and g.SP = W/16 + 2 <= 62: the random and edge inputs of
    test_gpu_ingest, ONT (N = 10k, W = 587, SP = 38) and 80-SNP reads, each into cleared counts and on top of them, on
    all SMs (148 CTAs), 2 and 3 SMs (one pair) and 1 SM (the single-CTA kernel)."""
    _run_fresh("_lumma_pairs", HX_LUMMA_PAIRS="1")


@pytest.mark.parametrize("read_w,rank_w", [(1, 0), (1, 1 << 20), (4096, 0), (4096, 1 << 20)])
def test_slice_weights(c_oracle, read_w, rank_w):
    """HX_UM_READ_W / HX_UM_RANK_W (read once per process) move k1_umma's slice cuts and its job-table bound `per`:
    with a read weight of 1 and a rank weight of 2^20 the bound from the weights alone is ~2e9 reads per CTA on the
    300k-site shape, where no slice can hold more than all the reads.  Kernels 2 and 5 slice with the built-in weights
    and run beside it as controls."""
    _run_fresh("_slice_weights", HX_UM_READ_W=str(read_w), HX_UM_RANK_W=str(rank_w))


def test_sorted_prefix_unsorted_tail(c_oracle):
    """250k reads, the first 60 % sorted by rank and the rest shuffled, in one ingest_packed: the host pipeline sends
    the sorted chunks in the dense encoding until a chunk is not sorted (HX_E_STATE), then hands the rest to the
    packed path.  The hand-back records that the process met unsorted input before the rest is launched, so in a
    fresh process too the auto kernel queues the counting-sort tensor-core kernel behind the sorted-run kernel; a
    fixed sorted-run kernel (6) queues one RED per pair instead.  All three runs equal the oracle."""
    _run_fresh("_sorted_prefix")
