"""Parity of the CUDA recovery path against the oracle: identical haplotypes, matrices after reweighting equal;
per-haplotype statistics bit for bit against the C oracle (removed mass within the rounding of its summation order,
same_stats) and within 1e-6 relative (north_star) against the Python goldens."""
import os

import numpy as np
import pytest

from gretel_b200 import synth
from oracle import hansel_oracle as o
from tests.test_gpu_recover_switches import same_stats

pytestmark = pytest.mark.gpu
RTOL = 1e-6          # north_star tolerance for per-haplotype likelihoods (log space)


def _mk(rank, off, codes, N, W, L=None, **kw):
    from gretel_b200 import util
    h = util.load_from_packed(rank, off, codes, N, band_w=W)
    if L is not None:
        h.L = L
    for k, v in kw.items():
        setattr(h, k, v)
    return h


@pytest.mark.parametrize("seed", range(6))
def test_small_against_literal_python_oracle(seed):
    """Everything the Hansel surface returns, on small dense cases, vs the literal oracle."""
    from gretel_b200 import gretel
    rng = np.random.default_rng(900 + seed)
    N = int(rng.integers(3, 14))
    rank, off, codes = synth.random_packed(rng, N, int(rng.integers(5, 60)), int(rng.integers(2, 8)),
                                           p_special=0.15)
    v_site = "to" if seed % 2 else "from"
    ho = o.load_from_packed(rank, off, codes, N, v_site=v_site)
    h = _mk(rank, off, codes, N, N + 1, v_site=v_site)
    assert (h.n_slices, h.n_crumbs, h.L) == (ho.n_slices, ho.n_crumbs, ho.L)
    assert np.array_equal(h.to_dense(), ho.m)
    for L in (1, 2, 5):
        h.L = ho.L = L
        for p in range(N + 1):
            assert h.get_counts_at(p) == ho.get_counts_at(p)
        # edge weights along the oracle's own greedy path
        path, _, _ = o.generate_path(N, ho, ho.copy())
        if path is None:
            continue
        for snp in range(1, N + 1):
            a, b = h.get_edge_weights_at(snp, path), ho.get_edge_weights_at(snp, path)
            assert list(a) == list(b)
            for k in a:
                assert a[k] == pytest.approx(b[k], rel=1e-12)
            assert h.get_marginal_of_at(path[snp], snp) == ho.get_marginal_of_at(path[snp], snp)
    h.L = ho.L = 3
    it_o, paths_o = o.recover(ho, N, max_paths=8)
    hc = h.copy()
    it_g, paths_g = gretel.recover(h, N, max_paths=8, resident=True)
    it_h, _ = gretel.recover(hc, N, max_paths=8, resident=False)
    for its in (it_g, it_h):
        assert [i["path"] for i in its] == [i["path"] for i in it_o]
        for a, b in zip(its, it_o):
            for key in ("hp_current", "hp_original", "min_marginal", "ratio", "removed"):
                assert a[key] == pytest.approx(b[key], rel=RTOL, abs=1e-12)
    assert list(paths_g) == list(paths_o)
    assert np.allclose(h.to_dense(), ho.m, rtol=1e-6, atol=0)
    assert np.array_equal(hc.to_dense(), h.to_dense())


@pytest.mark.parametrize("name,n_reads,L", [("hiv", 20_000, None), ("hiv", 20_000, 1), ("hiv", 20_000, 8),
                                            ("metagenome", 200_000, None), ("ont", 300, 6), ("ont", 300, None)])
def test_workload_recovery_against_c_oracle(c_oracle, name, n_reads, L):
    from gretel_b200 import gretel
    w = synth.scaled(synth.WORKLOADS[name], n_reads)
    d = synth.generate(w)
    N, W = w.n_snps, d["max_k"] - 1
    band, totals = c_oracle.ingest(d["rank"], d["off"], d["codes"], N, W)
    h = _mk(d["rank"], d["off"], d["codes"], N, W)
    if L is None:
        L = h.L
    h.L = L
    cur = band.astype(np.float32)
    orig = cur.copy()
    # the synthetic region may contain uncovered sites: then both sides must report the same hole
    exp = []
    for it in range(6):
        pc, res = c_oracle.generate_path(cur, orig, N, W, L)
        if pc is None:
            exp.append(("hole", res))
            break
        ratio = max(res[2], 0.01)
        removed = c_oracle.reweight_path(cur, N, W, pc, ratio)
        exp.append((pc, res, ratio, removed))
    orig_h = h.copy()
    got = []
    for it in range(6):
        r = h.generate_path_codes(orig_h)
        if r[0] is None:
            got.append(("hole", r[1]))
            break
        ratio = max(r[3], 0.01)
        got.append((r[0], r[1:], ratio, h.reweight_path_codes(r[0], ratio)))
    assert len(got) == len(exp)
    for g, e in zip(got, exp):
        if isinstance(e[0], str):
            assert g == e
            continue
        assert np.array_equal(g[0], e[0])
        same_stats(g[1] + (g[2], g[3]), e[1] + (e[2], e[3]), N, W)
    assert np.array_equal(h.band(), cur)


def test_hole_reported():
    """gretel.py:176-180: a site with no evidence ends recovery with (None, None, None)."""
    from gretel_b200 import gretel
    rank = np.array([0, 3], np.int32)
    off = np.array([0, 2, 4], np.int64)
    codes = np.array([0, 1, 2, 3], np.uint8)          # sites 1,2 and 4,5 bridged; site 3 is not
    h = _mk(rank, off, codes, 5, 6)
    assert gretel.gap_check(h, 5) == [2, 3]      # site 5 carries the end sentinel (util.py:271-275)
    assert gretel.generate_path(5, h, h.copy()) == (None, None, None)
    its, paths = gretel.recover(h, 5, max_paths=3)
    assert its == [] and paths == {}


def test_recover_terminates_when_evidence_is_spent():
    """A single-strain region: marginals are 1.0, the ratio is 1.0, everything is removed
    and the second generate_path finds a hole."""
    from gretel_b200 import gretel
    N = 6
    rank = np.zeros(4, np.int32)
    off = np.arange(0, 4 * N + 1, N).astype(np.int64)
    codes = np.tile(np.array([0, 1, 2, 3, 0, 1], np.uint8), 4)
    h = _mk(rank, off, codes, N, N + 1)
    ho = o.load_from_packed(rank, off, codes, N)
    it_o, _ = o.recover(ho, N, max_paths=5)
    it_g, _ = gretel.recover(h, N, max_paths=5)
    assert [i["path"] for i in it_g] == [i["path"] for i in it_o] and len(it_g) >= 1
    for a, b in zip(it_g, it_o):
        assert a["removed"] == pytest.approx(b["removed"], rel=1e-9)


def _walk_vs_c_oracle(c_oracle, h, band, N, W, L, iters=3, packed=None):
    cur, orig = band.astype(np.float32).copy(), band.astype(np.float32).copy()
    h.L = L
    orig_h = h.copy()
    for it in range(iters):
        pc, res = c_oracle.generate_path(cur, orig, N, W, L)
        r = h.generate_path_codes(orig_h)
        if pc is None:
            assert r[0] is None and r[1] == res
            return
        assert r[0] is not None
        assert np.array_equal(r[0], pc), "L=%d iteration %d" % (L, it)      # sequences identical, ties included
        ratio = max(res[2], 0.01)
        removed = h.reweight_path_codes(r[0], ratio)
        same_stats(r[1:] + (ratio, removed), res + (ratio, c_oracle.reweight_path(cur, N, W, pc, ratio)), N, W,
                   "L=%d iteration %d" % (L, it))
    assert np.array_equal(h.band(), cur)


@pytest.mark.parametrize("L", list(range(1, 35)) + [40, 47])
def test_every_lookback_depth(c_oracle, L):
    """One case per lookback depth: each instantiation of the fixed-point walk (L <= 32 inside the band), the
    staged float64 walk beyond it and lookbacks that leave the band.  Thin random evidence gives many exact ties,
    so the exact re-evaluation (first maximum wins, gretel.py:166-174) is exercised at every depth - including
    candidates that tie in real arithmetic, where the pick hangs on the last bit of log10 / 10**x: the kernels
    evaluate both exactly as the host's libm does (test_device_math_is_the_hosts_libm), so no divergence is allowed."""
    rng = np.random.default_rng(4200 + L)
    N = 150
    rank, off, codes = synth.random_packed(rng, N, 900, 38, p_special=0.05)
    W = int(np.diff(off).max()) - 1
    band, _ = c_oracle.ingest(rank, off, codes, N, W)
    h = _mk(rank, off, codes, N, W)
    _walk_vs_c_oracle(c_oracle, h, band, N, W, L, packed=(rank, off, codes))


def test_walk_leaves_fixed_point_range(c_oracle):
    """Counts so large that a log10 term does not fit the fixed-point table: the walk must notice and decide
    every site from the float64 terms."""
    rng = np.random.default_rng(77)
    N = 60
    rank, off, codes = synth.random_packed(rng, N, 600, 12, p_special=0.05)
    W = int(np.diff(off).max()) - 1
    band, _ = c_oracle.ingest(rank, off, codes, N, W)
    band = band.astype(np.float32)
    band[band > 0] *= np.float32(1e17)
    band[10:50:7] *= np.float32(1e3)
    h = _mk(rank, off, codes, N, W)
    h.load_band(band)
    _walk_vs_c_oracle(c_oracle, h, band, N, W, 6, iters=2)


def _float64_walk(W, L):
    """Which float64 walk launch_generate runs for L > 32: k_walk_wide when three staged chunks of one site's tables
    (Lw * 448 + 64 bytes, Lw = min(L, W)) cannot fit its 200 KiB of shared memory, k_walk_tables otherwise."""
    Lw = min(L, W)
    return "wide" if (200 * 1024) // (3 * (Lw * 448 + 64)) < 1 else "tables"


@pytest.mark.parametrize("kernel,dL", [("tables", None), ("wide", 0), ("wide", 20)],
                         ids=["tables_L100", "wide_L_W", "wide_L_W+20"])
def test_wide_band_walks(c_oracle, kernel, dL):
    """Reads of up to 170 SNPs make a band wide enough (W >= 153) that one site's float64 tables do not fit the staged
    walk: k_walk_wide walks at L = W, and at L = W + 20 with lookbacks beyond the band (log10(1/V) terms).  L = 100
    is the staged k_walk_tables inside the same band."""
    rng = np.random.default_rng(5150)
    N = 400
    rank, off, codes = synth.random_packed(rng, N, 600, 170, p_special=0.05)
    W = int(np.diff(off).max()) - 1
    L = 100 if dL is None else W + dL
    assert W >= 153 and _float64_walk(W, L) == kernel and (L > W) == (dL == 20)
    band, _ = c_oracle.ingest(rank, off, codes, N, W)
    cur = band.astype(np.float32)
    assert c_oracle.generate_path(cur, cur.copy(), N, W, L)[0] is not None      # the first walk reaches site N
    h = _mk(rank, off, codes, N, W)
    _walk_vs_c_oracle(c_oracle, h, band, N, W, L, packed=(rank, off, codes))


import glob

GOLDEN_RECOVERY = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "ref_recovery_*.npz")))


@pytest.mark.parametrize("path", GOLDEN_RECOVERY, ids=[os.path.basename(p)[:-4] for p in GOLDEN_RECOVERY])
@pytest.mark.parametrize("resident", [True, False])
def test_gpu_against_reference_code_golden(path, resident):
    """Golden vectors made by the reference's own generate_path / reweight_hansel_from_path
    (tests/golden/make_golden.py): identical haplotypes, likelihoods within 1e-6 relative."""
    from gretel_b200 import gretel
    z = np.load(path)
    N, L, v_site = int(z["N"]), int(z["L"]), str(z["v_site"])
    h = _mk(z["rank"], z["off"], z["codes"], N, N + 1, L=L, v_site=v_site)
    assert (h.n_slices, h.n_crumbs) == (int(z["n_slices"]), int(z["n_crumbs"]))
    assert np.array_equal(h.to_dense(), z["dense_before"])
    its, _ = gretel.recover(h, N, max_paths=len(z["paths"]), resident=resident)
    assert len(its) == len(z["paths"])
    for it, gp, gs in zip(its, z["paths"], z["stats"]):
        assert list(h.encode_path(it["hansel_path"])) == list(gp)
        for got, exp in zip((it["hp_current"], it["hp_original"], it["min_marginal"], it["ratio"], it["removed"]), gs):
            assert got == pytest.approx(exp, rel=RTOL, abs=1e-12)
    assert np.allclose(h.to_dense(), z["dense_after"], rtol=1e-6, atol=0)


def test_device_math_is_the_hosts_libm():
    """log10 and 10**x on the device (glibc_math.cuh, a transcription of this image's glibc) equal the host's libm -
    what math.log10 and float ** reach in the reference (gretel.py:166-187) - bit for bit on two million arguments each."""
    import ctypes as C
    import math
    from gretel_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(12345)
    n = 250_000
    xs = np.concatenate([
        rng.random(n),                                                        # probabilities
        (1.0 + rng.integers(0, 100000, n)) / (1.0 + rng.integers(0, 200000, n) + rng.integers(0, 100000, n)),
        1.0 + (rng.random(n) - 0.5) * 0.2,                                    # around 1
        np.exp((rng.random(n) - 0.5) * 1400.0),                               # the whole range
        1.0 / rng.integers(1, 64, n),
        rng.integers(1, 10**6, n).astype(np.float64),
        np.maximum(rng.random(n) * 1e-310, 5e-324),                           # subnormal
        np.ldexp(1.0 + rng.random(n), rng.integers(-1022, 1023, n)),
    ]).astype(np.float64)
    ys = np.concatenate([-rng.random(4 * n) * 330.0, -rng.random(2 * n) * 20.0, (rng.random(n) - 0.5) * 600.0,
                         (rng.random(n // 2) - 0.5) * 1e-3, -rng.random(n // 4) * 1e-20, -307.0 - rng.random(n // 4) * 20.0,
                         np.zeros(4)]).astype(np.float64)
    for which, arg, fn in ((0, xs, math.log10), (1, ys, lambda v: 10.0 ** v)):
        out = np.empty_like(arg)
        _lib.check(lib.hx_device_math(0, which, arg.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), len(arg)))
        want = np.array([fn(float(v)) for v in arg], dtype=np.float64)
        bad = np.flatnonzero(out.view(np.uint64) != want.view(np.uint64))
        assert bad.size == 0, (which, arg[bad[:5]], out[bad[:5]], want[bad[:5]])
